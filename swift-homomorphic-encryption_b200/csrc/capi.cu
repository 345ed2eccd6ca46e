// capi.cu -- the C ABI declared in include/hecuda.h.  No torch types, no exceptions across the boundary.
//
// Host-pointer entry points run a chunked, double-buffered pipeline (two workspaces on two streams) so that the
// H2D copy of chunk k+1, the kernels of chunk k and the D2H copy of chunk k-1 overlap when the caller's buffers are
// pinned.  Device-pointer entry points enqueue on the caller's stream and do not synchronize.
#include "../../include/hecuda.h"

#include <cuda_runtime.h>
#include <sched.h>
#include <sys/syscall.h>
#include <unistd.h>

#include <algorithm>
#include <cctype>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <initializer_list>
#include <map>
#include <memory>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "capi_internal.hpp"

namespace hecuda {
std::atomic<unsigned long long> g_kernel_launches{0};
}

using namespace hecuda;

namespace hecuda {
namespace api {

static thread_local std::string tl_error;

int32_t fail(int32_t code, const std::string &msg) {
    tl_error = msg;
    return code;
}
int32_t cuda_fail(cudaError_t e, const char *what) {
    return fail(HECUDA_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}
const char *last_error_cstr() { return tl_error.c_str(); }

}  // namespace api
}  // namespace hecuda

using namespace hecuda::api;

namespace hecuda {
namespace api {

cudaError_t wait_stream(cudaStream_t s) {
    // Default: yield the CPU while waiting (an event created with cudaEventBlockingSync).  Spinning in
    // cudaStreamSynchronize burns a core per waiting thread; with many serving threads inside a CPU-quota'd container
    // the spinners get throttled and throughput collapses (measured: 8-32 PIR threads under a 16-core quota swing
    // between 370 and 1100 queries/s spinning, 1000-1135 blocking).  HECUDA_BLOCKING_SYNC=0 restores the spin wait.
    static const bool blocking = [] {
        const char *env = std::getenv("HECUDA_BLOCKING_SYNC");
        return !(env && env[0] == '0');
    }();
    if (!blocking) return cudaStreamSynchronize(s);
    thread_local cudaEvent_t event = nullptr;
    thread_local int event_device = -1;
    int device = 0;
    cudaError_t e = cudaGetDevice(&device);
    if (e != cudaSuccess) return e;
    if (!event || event_device != device) {
        if ((e = cudaEventCreateWithFlags(&event, cudaEventBlockingSync | cudaEventDisableTiming)) != cudaSuccess) return e;
        event_device = device;
    }
    if ((e = cudaEventRecord(event, s)) != cudaSuccess) return e;
    return cudaEventSynchronize(event);
}

int32_t check_ctx(const hecuda_context *h) {
    if (!h || !h->ctx) return fail(HECUDA_ERR_INVALID_ARGUMENT, "invalidContext: null context");
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess) return fail(HECUDA_ERR_NO_DEVICE, "no CUDA device available");
    if (dev != h->ctx->device) {
        cudaError_t e = cudaSetDevice(h->ctx->device);
        if (e != cudaSuccess) return cuda_fail(e, "cudaSetDevice");
    }
    return HECUDA_OK;
}

bool make_map(const Context &c, int32_t base, int32_t rows, NttRowMap &map, std::string &err) {
    switch (base) {
        case HECUDA_BASE_Q:
            if (rows < 1 || rows > c.L) { err = "invalidPolyContext: row_count must be in [1, L] for BASE_Q"; return false; }
            map = c.map_q(rows);
            return true;
        case HECUDA_BASE_Q_BSK:
            if (rows != 2 * c.L + 1) { err = "invalidPolyContext: BASE_Q_BSK needs 2L+1 rows"; return false; }
            map = c.map_qbsk();
            return true;
        case HECUDA_BASE_Q_AUX:
            if (rows != 2 * c.L + 1) { err = "invalidPolyContext: BASE_Q_AUX needs 2L+1 rows"; return false; }
            map = c.map_qaux();
            return true;
        case HECUDA_BASE_KEYSWITCH:
            if (!c.has_ks) { err = "invalidPolyContext: these parameters have no key-switching modulus"; return false; }
            if (rows < 2 || rows > c.L + 1) { err = "invalidPolyContext: BASE_KEYSWITCH needs 2..L+1 rows"; return false; }
            map = c.map_ks(rows - 1);
            return true;
        default:
            err = "invalidPolyContext: unknown base";
            return false;
    }
}

// ---------------------------------------------------------------- device-side op bodies (enqueue only)

// scratch words needed per ciphertext pair / ciphertext
size_t multiply_scratch_words(const Context &c) { return (size_t)7 * (2 * c.L + 1) * c.n; }
size_t relinearize_scratch_words(const Context &c, int l) { return (size_t)((l + 1) * l + 2 * (l + 1)) * c.n; }

cudaError_t multiply_chunk(const Context &c, u64 *scratch, const u64 *lhs, const u64 *rhs, u64 *out, int64_t items,
                           cudaStream_t s) {
    const int R = 2 * c.L + 1;
    const size_t poly_words = (size_t)R * c.n;
    cudaError_t e;
    u64 *ext = scratch, *ten = scratch + 4 * poly_words * items;
    const NttRowMap map = c.map_qaux();
    // computeBehzPolys for both operands: lift + forward NTT      (Bfv+Multiply.swift:51-57)
    if ((e = launch_lift(c, lhs, 2, ext, 4, 0, items, s)) != cudaSuccess) return e;
    if ((e = launch_lift(c, rhs, 2, ext, 4, 2, items, s)) != cudaSuccess) return e;
    if ((e = launch_ntt_forward(c, map, ext, ext, items * 4 * R, s)) != cudaSuccess) return e;
    // tensor product                                               (Bfv+Multiply.swift:80-82)
    if ((e = launch_tensor(c, ext, ten, items, s)) != cudaSuccess) return e;
    // dropExtendedBase: (* t) folded into the inverse NTT, floor    (Bfv+Multiply.swift:31-48)
    if ((e = launch_ntt_inverse(c, map, ten, ten, items * 3 * R, kScaleTMont, s)) != cudaSuccess) return e;
    return launch_floor(c, ten, out, items * 3, s);
}

// _computeKeySwitchingUpdate (Bfv+Keys.swift:123-208) of `target` (l rows per item, items `target_stride` words apart)
// + the caller's accumulation: out[item][c] = update[c] (+ base[item][c] for the components in base_mask).
cudaError_t keyswitch_chunk(const Context &c, u64 *scratch, const u64 *key, const u64 *target, int64_t target_stride,
                            int l, const u64 *base, int64_t base_stride, int base_mask, u64 *out, int64_t items,
                            cudaStream_t s) {
    const size_t dig_words = (size_t)(l + 1) * l * c.n;
    cudaError_t e;
    u64 *dig = scratch, *prod = scratch + dig_words * items;
    // digits: forward NTT that gathers [target row j]_{m_r} straight from the source      (Bfv+Keys.swift:165-179)
    if ((e = launch_ntt_forward(c, c.map_ks_digits(l, target_stride), target, dig, items * (l + 1) * l, s)) != cudaSuccess)
        return e;
    if ((e = launch_ks_mac(c, dig, key, l, prod, items, s)) != cudaSuccess) return e;
    if ((e = launch_ntt_inverse(c, c.map_ks(l), prod, prod, items * 2 * (l + 1), kScaleMont, s)) != cudaSuccess) return e;
    return launch_ks_finish(c, prod, base, base_stride, base_mask, l, out, items, s);
}

// Bfv.relinearize (Bfv.swift:201-219): key-switch poly 2, add the update to polys 0 and 1
cudaError_t relinearize_chunk(const Context &c, u64 *scratch, const u64 *key, const u64 *ct3, int l, u64 *out,
                              int64_t items, cudaStream_t s) {
    const int64_t ct_stride = (int64_t)3 * l * c.n;
    return keyswitch_chunk(c, scratch, key, ct3 + (int64_t)2 * l * c.n, ct_stride, l, ct3, ct_stride, 3, out, items, s);
}

// Bfv.applyGalois (Bfv.swift:174-198): c0' = galois(c0) + update[0], c1' = update[1], update = keyswitch(galois(c1))
size_t galois_scratch_words(const Context &c, int l) { return relinearize_scratch_words(c, l) + (size_t)l * c.n; }
cudaError_t apply_galois_chunk(const Context &c, u64 *scratch, const u64 *key, const u64 *ct, int l, unsigned element,
                               u64 *out, int64_t items, cudaStream_t s) {
    const int64_t poly = (int64_t)l * c.n, ct_stride = 2 * poly;
    u64 *perm1 = scratch;                      // items x l x N
    u64 *ks_scratch = scratch + poly * items;
    const NttRowMap map = c.map_q(l);
    cudaError_t e;
    if ((e = launch_galois_coeff(c, map, element, ct, ct_stride, out, ct_stride, items, s)) != cudaSuccess) return e;
    if ((e = launch_galois_coeff(c, map, element, ct + poly, ct_stride, perm1, poly, items, s)) != cudaSuccess) return e;
    return keyswitch_chunk(c, ks_scratch, key, perm1, poly, l, out, ct_stride, 1, out, items, s);
}

// Bfv.innerProduct(_:_:) (Bfv.swift:315-361): sum of the tensor products of `pairs` ciphertext pairs in [Q, Bsk],
// then ONE dropExtendedBase -- instead of `pairs` full multiplies.
cudaError_t inner_product_chunk(const Context &c, u64 *scratch, const u64 *lhs, const u64 *rhs, int64_t pairs,
                                       u64 *out, int64_t groups, cudaStream_t s) {
    const int R = 2 * c.L + 1;
    const size_t poly_words = (size_t)R * c.n;
    const int64_t items = groups * pairs;
    u64 *ext = scratch, *ten = scratch + 4 * poly_words * items;
    const NttRowMap map = c.map_qaux();
    cudaError_t e;
    if ((e = launch_lift(c, lhs, 2, ext, 4, 0, items, s)) != cudaSuccess) return e;
    if ((e = launch_lift(c, rhs, 2, ext, 4, 2, items, s)) != cudaSuccess) return e;
    if ((e = launch_ntt_forward(c, map, ext, ext, items * 4 * R, s)) != cudaSuccess) return e;
    if ((e = launch_tensor_sum(c, ext, ten, pairs, groups, s)) != cudaSuccess) return e;
    if ((e = launch_ntt_inverse(c, map, ten, ten, groups * 3 * R, kScaleTMont, s)) != cudaSuccess) return e;
    return launch_floor(c, ten, out, groups * 3, s);
}
size_t inner_product_scratch_words(const Context &c, int64_t pairs) {
    return (size_t)(4 * pairs + 3) * (2 * c.L + 1) * c.n;
}

}  // namespace api
}  // namespace hecuda

namespace {

// Where the buffers of a batched call live and how wide their words are.  Host64 / Host32 run the double-buffered host
// pipeline; Host32 buffers hold uint32 words (Bfv<UInt32>), widened after each H2D copy and narrowed before each D2H
// copy.  Device buffers are uint64 on the device, enqueued on the caller's stream.
enum class Io { Host64, Host32, Device };

// A caller buffer of `words_per_item` words per batch item.
struct Operand {
    const u64 *src;
    size_t words_per_item;
};

// One chunk of a batched call: items [first, first + items) of the batch, on device buffers.
struct Chunk {
    u64 *scratch;  // the op's scratch words per item x items
    const u64 *in[2];
    u64 *out;
    int64_t first, items;
    cudaStream_t stream;
};

// Generic double-buffered host pipeline: for each chunk, copy inputs in, run `body`, copy outputs out.
template <class Body>
int32_t host_pipeline(const hecuda_context *h, bool io32, int64_t batch, int64_t chunk_hint, size_t scratch_words_per_item,
                      std::initializer_list<Operand> inputs, u64 *host_out, size_t out_words_per_item, Body body) {
    if (batch == 0) return HECUDA_OK;
    // `depth` stages in flight, each on its own stream: H2D of stage k+1.., kernels of stage k, D2H of stage k-1
    static const int depth = [] {
        const char *env = std::getenv("HECUDA_PIPELINE_DEPTH");
        const int d = env ? std::atoi(env) : 3;
        return d < 1 ? 1 : (d > 8 ? 8 : d);
    }();
    static const int64_t min_stages = [] {
        const char *env = std::getenv("HECUDA_PIPELINE_STAGES");
        const long long v = env ? std::atoll(env) : 16;
        return (int64_t)(v < 1 ? 1 : v);
    }();
    std::vector<std::unique_ptr<WsGuard>> guards;
    std::vector<Workspace *> ws;
    for (int i = 0; i < depth; ++i) {
        guards.emplace_back(new WsGuard(h));
        if (!guards.back()->w) return fail(HECUDA_ERR_CUDA, "could not create a CUDA stream / workspace");
        ws.push_back(guards.back()->w);
    }
    int64_t chunk = std::max<int64_t>(1, std::min<int64_t>(chunk_hint, batch));
    if (batch >= 64) chunk = std::min<int64_t>(chunk, std::max<int64_t>(16, (batch + min_stages - 1) / min_stages));
    // On any early return, earlier stages may still have copies into / out of the caller's buffers in flight on the
    // other streams: wait for all of them so the caller may free or reuse its buffers as soon as it sees the error.
    struct DrainOnExit {
        std::vector<Workspace *> &ws;
        ~DrainOnExit() {
            for (Workspace *w : ws) wait_stream(w->stream);
        }
    } drain{ws};
    int k = 0;
    for (int64_t done = 0; done < batch; done += chunk, ++k) {
        Workspace &w = *ws[k % depth];
        const int64_t items = std::min<int64_t>(chunk, batch - done);
        // Work on one workspace is ordered by its stream; buffers only ever grow (first `depth` iterations).
        // slot 0 = kernel scratch, slot 4 = staged inputs (back to back), slot 5 = staged output
        size_t in_words = 0;
        for (const Operand &io : inputs) in_words += io.words_per_item * (size_t)items;
        const size_t out_words = out_words_per_item * (size_t)items;
        CK(w.reserve(0, scratch_words_per_item * (size_t)items));
        CK(w.reserve(4, in_words));
        CK(w.reserve(5, out_words));
        if (io32) {  // slots 6 / 7: the uint32 images (each input starts on a 16-byte boundary)
            CK(w.reserve(6, in_words / 2 + inputs.size() * 2 + 2));
            CK(w.reserve(7, out_words / 2 + 2));
        }
        Chunk c{w.buf[0], {nullptr, nullptr}, w.buf[5], done, items, w.stream};
        size_t off = 0, off32 = 0;
        int i = 0;
        for (const Operand &io : inputs) {
            const size_t words = io.words_per_item * (size_t)items;
            if (io32) {
                u32 *raw = reinterpret_cast<u32 *>(w.buf[6]) + off32;
                CK(cudaMemcpyAsync(raw, reinterpret_cast<const u32 *>(io.src) + io.words_per_item * (size_t)done,
                                   words * sizeof(u32), cudaMemcpyHostToDevice, w.stream));
                CK(launch_widen(raw, w.buf[4] + off, (int64_t)words, w.stream));
                off32 += (words + 3) & ~(size_t)3;
            } else {
                CK(cudaMemcpyAsync(w.buf[4] + off, io.src + io.words_per_item * (size_t)done, words * sizeof(u64),
                                   cudaMemcpyHostToDevice, w.stream));
            }
            c.in[i++] = w.buf[4] + off;
            off += words;
        }
        cudaError_t e = body(c);
        if (e != cudaSuccess) return cuda_fail(e, "kernel launch");
        if (io32) {
            CK(launch_narrow(w.buf[5], reinterpret_cast<u32 *>(w.buf[7]), (int64_t)out_words, w.stream));
            CK(cudaMemcpyAsync(reinterpret_cast<u32 *>(host_out) + out_words_per_item * (size_t)done, w.buf[7],
                               out_words * sizeof(u32), cudaMemcpyDeviceToHost, w.stream));
        } else {
            CK(cudaMemcpyAsync(host_out + out_words_per_item * (size_t)done, w.buf[5], out_words * sizeof(u64),
                               cudaMemcpyDeviceToHost, w.stream));
        }
    }
    for (Workspace *w : ws) CK(wait_stream(w->stream));
    return HECUDA_OK;
}

// Runs `body` over a batch of `batch` items held in `io`'s buffers.  Host calls go through the host pipeline, which
// stages at most `chunk_hint` items at a time.  Device calls enqueue on `stream` and do not synchronise (so they can
// be captured in a graph): ops with scratch run in chunks of min(chunk_hint, batch) items over one stream-ordered
// allocation, scratch-free ops run the whole batch in one pass.  `what` names a failed device launch.
template <class Body>
int32_t dispatch(const hecuda_context *h, Io io, void *stream, const char *what, int64_t batch, int64_t chunk_hint,
                 size_t scratch_words_per_item, std::initializer_list<Operand> inputs, void *out, size_t out_words_per_item,
                 Body body) {
    if (io != Io::Device)
        return host_pipeline(h, io == Io::Host32, batch, chunk_hint, scratch_words_per_item, inputs, (u64 *)out,
                             out_words_per_item, body);
    if (batch == 0) return HECUDA_OK;
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t chunk = scratch_words_per_item ? std::max<int64_t>(1, std::min<int64_t>(chunk_hint, batch)) : batch;
    u64 *scratch = nullptr;
    if (scratch_words_per_item) CK(cudaMallocAsync(&scratch, scratch_words_per_item * (size_t)chunk * sizeof(u64), s));
    cudaError_t e = cudaSuccess;
    for (int64_t first = 0; first < batch && e == cudaSuccess; first += chunk) {
        Chunk c{scratch, {nullptr, nullptr}, (u64 *)out + out_words_per_item * first, first,
                std::min<int64_t>(chunk, batch - first), s};
        int i = 0;
        for (const Operand &io : inputs) c.in[i++] = io.src + io.words_per_item * first;
        e = body(c);
    }
    if (scratch) {
        const cudaError_t f = cudaFreeAsync(scratch, s);
        if (e == cudaSuccess && f != cudaSuccess) return cuda_fail(f, "cudaFreeAsync(scratch, s)");
    }
    return e == cudaSuccess ? HECUDA_OK : cuda_fail(e, what);
}

// uint32 buffers need a context made by hecuda_context_create_u32 (its m~, gamma and Bsk).
int32_t need_word32(const hecuda_context *h) {
    if (!h || !h->ctx) return fail(HECUDA_ERR_INVALID_ARGUMENT, "invalidContext: null context");
    if (h->ctx->word_bits != 32) return fail(HECUDA_ERR_INVALID_ARGUMENT, "invalidContext: not a Bfv<UInt32> context (hecuda_context_create_u32)");
    return HECUDA_OK;
}

// The first check of every batched call: the Host32 precondition, then the context.
int32_t check_io(const hecuda_context *h, Io io) {
    if (io == Io::Host32) {
        int32_t rc = need_word32(h);
        if (rc) return rc;
    }
    return check_ctx(h);
}

// The evaluation key of a call is present (for relinearization: filled in) and belongs to the call's context.
int32_t check_key(const hecuda_context *h, const hecuda_evk *k, bool relin) {
    if (!k || (relin && !k->loaded)) return fail(HECUDA_ERR_MISSING_KEY, relin ? "missingRelinearizationKey" : "missingGaloisKey");
    if (k->owner != h) return fail(HECUDA_ERR_INVALID_ARGUMENT, "invalidContext: evaluation key belongs to another context");
    return HECUDA_OK;
}

// 1 <= l <= L; `kind` is the error's prefix (invalidCiphertext / invalidPolyContext).
int32_t check_level(const hecuda_context *h, int32_t l, const char *kind) {
    if (l < 1 || l > h->ctx->L) return fail(HECUDA_ERR_INVALID_ARGUMENT, std::string(kind) + ": moduli_count out of range");
    return HECUDA_OK;
}

// A batch size is not negative, and a non-empty batch has every buffer.
int32_t check_batch(int64_t batch, std::initializer_list<const void *> buffers, const char *msg) {
    bool missing = false;
    for (const void *p : buffers) missing |= !p;
    if (batch < 0 || (batch && missing)) return fail(HECUDA_ERR_INVALID_ARGUMENT, msg);
    return HECUDA_OK;
}

// Items per host-pipeline stage for a scratch-free op: ~4 M words (32 MB) of `words_per_item`-word items per stage.
int64_t stage_items(size_t words_per_item, size_t stage_words = (size_t)4 * 1024 * 1024) {
    return std::max<int64_t>(1, (int64_t)(stage_words / std::max<size_t>(1, words_per_item)));
}

}  // namespace

// ====================================================================================================== C ABI

extern "C" {

int32_t hecuda_version(void) { return 100; }
const char *hecuda_last_error(void) { return last_error_cstr(); }

int32_t hecuda_device_count(int32_t *count) {
    if (!count) return fail(HECUDA_ERR_INVALID_ARGUMENT, "null count");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        *count = 0;
        return fail(HECUDA_ERR_NO_DEVICE, std::string("no CUDA device: ") + cudaGetErrorString(e));
    }
    *count = n;
    return HECUDA_OK;
}
int32_t hecuda_set_device(int32_t device) {
    CK(cudaSetDevice(device));
    return HECUDA_OK;
}

// NUMA placement of the host side of one GPU: pin the calling thread (threads it creates later inherit the mask) to the
// CPUs local to the GPU's PCIe root and prefer that node for page allocations, so that pinned staging buffers
// allocated afterwards (hecuda_host_alloc) and the copies out of them do not cross the socket interconnect.
int32_t hecuda_bind_host_to_device(int32_t device, int32_t *numa_node, int32_t *cpu_count) {
    if (numa_node) *numa_node = -1;
    if (cpu_count) *cpu_count = 0;
    char bus[32] = {0};
    CK(cudaDeviceGetPCIBusId(bus, sizeof(bus), device));
    for (char *c = bus; *c; ++c) *c = (char)std::tolower((unsigned char)*c);
    const std::string dir = std::string("/sys/bus/pci/devices/") + bus + "/";
    int node = -1;
    if (FILE *f = std::fopen((dir + "numa_node").c_str(), "r")) {
        if (std::fscanf(f, "%d", &node) != 1) node = -1;
        std::fclose(f);
    }
    char list[4096] = {0};
    if (FILE *f = std::fopen((dir + "local_cpulist").c_str(), "r")) {
        if (!std::fgets(list, sizeof(list), f)) list[0] = 0;
        std::fclose(f);
    }
    cpu_set_t current, want;
    CPU_ZERO(&want);
    if (sched_getaffinity(0, sizeof(current), &current) != 0) return HECUDA_OK;  // nothing to intersect with: leave as is
    int picked = 0;
    char *save = nullptr;
    for (char *tok = strtok_r(list, ",\n", &save); tok; tok = strtok_r(nullptr, ",\n", &save)) {
        int lo = 0, hi = 0;
        const int fields = std::sscanf(tok, "%d-%d", &lo, &hi);
        if (fields < 1) continue;
        if (fields == 1) hi = lo;
        for (int c = lo; c <= hi && c < CPU_SETSIZE; ++c)
            if (CPU_ISSET(c, &current)) {
                CPU_SET(c, &want);
                ++picked;
            }
    }
    if (picked > 0) sched_setaffinity(0, sizeof(want), &want);
    if (node >= 0 && node < 64) {  // MPOL_PREFERRED: fall back to other nodes rather than fail when the node is full
        unsigned long mask = 1ul << node;
        syscall(SYS_set_mempolicy, 1 /* MPOL_PREFERRED */, &mask, sizeof(mask) * 8);
    }
    if (numa_node) *numa_node = node;
    if (cpu_count) *cpu_count = picked;
    return HECUDA_OK;
}

int32_t hecuda_host_alloc(void **ptr, uint64_t bytes) {
    if (!ptr) return fail(HECUDA_ERR_INVALID_ARGUMENT, "null ptr");
    CK(cudaHostAlloc(ptr, bytes, cudaHostAllocDefault));
    return HECUDA_OK;
}
int32_t hecuda_host_free(void *ptr) {
    CK(cudaFreeHost(ptr));
    return HECUDA_OK;
}
int32_t hecuda_host_register(void *ptr, uint64_t bytes) {
    CK(cudaHostRegister(ptr, bytes, cudaHostRegisterDefault));
    return HECUDA_OK;
}
int32_t hecuda_host_unregister(void *ptr) {
    CK(cudaHostUnregister(ptr));
    return HECUDA_OK;
}

static int32_t context_create(int64_t poly_degree, const uint64_t *coefficient_moduli, int32_t moduli_count,
                              uint64_t plaintext_modulus, int word_bits, hecuda_context **out);
int32_t hecuda_context_create(int64_t poly_degree, const uint64_t *coefficient_moduli, int32_t moduli_count,
                              uint64_t plaintext_modulus, hecuda_context **out) {
    return context_create(poly_degree, coefficient_moduli, moduli_count, plaintext_modulus, 64, out);
}
int32_t hecuda_context_create_u32(int64_t poly_degree, const uint32_t *coefficient_moduli, int32_t moduli_count,
                                  uint32_t plaintext_modulus, hecuda_context **out) {
    if (!coefficient_moduli || moduli_count < 0) return fail(HECUDA_ERR_INVALID_ARGUMENT, "null argument");
    std::vector<uint64_t> wide(coefficient_moduli, coefficient_moduli + moduli_count);
    return context_create(poly_degree, wide.data(), moduli_count, plaintext_modulus, 32, out);
}
int32_t hecuda_context_word_bits(const hecuda_context *h, int32_t *bits) {
    if (!h || !bits) return fail(HECUDA_ERR_INVALID_ARGUMENT, "null argument");
    *bits = h->ctx->word_bits;
    return HECUDA_OK;
}
static int32_t context_create(int64_t poly_degree, const uint64_t *coefficient_moduli, int32_t moduli_count,
                              uint64_t plaintext_modulus, int word_bits, hecuda_context **out) {
    if (!out || !coefficient_moduli) return fail(HECUDA_ERR_INVALID_ARGUMENT, "null argument");
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(HECUDA_ERR_NO_DEVICE, "no CUDA device: libhecuda has no CPU fallback");
    std::string err;
    Context *c = Context::create(poly_degree, (const u64 *)coefficient_moduli, moduli_count, plaintext_modulus, err, word_bits);
    if (!c) {
        const bool unsupported = err.rfind("unsupported", 0) == 0;
        return fail(unsupported ? HECUDA_ERR_UNSUPPORTED : HECUDA_ERR_INVALID_ARGUMENT, err);
    }
    hecuda_context *h = new (std::nothrow) hecuda_context();
    if (!h) {
        delete c;
        return fail(HECUDA_ERR_CUDA, "out of host memory");
    }
    h->ctx = c;
    {   // keep stream-ordered scratch cached in the default pool instead of returning it to the OS at every sync
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, c->device) == cudaSuccess) {
            unsigned long long threshold = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &threshold);
        }
    }
    // pipeline stage size: keep one stage's intermediates (7 R N words per ciphertext pair) near the L2 size
    // Every kernel on this path is instruction-issue bound, not HBM bound (DESIGN.md), so large launches that
    // amortise wave tails beat L2-resident small ones: size a stage to ~2 GB of scratch.
    const size_t per_item = (size_t)7 * (2 * c->L + 1) * c->n * sizeof(u64);
    int64_t chunk = (int64_t)((size_t)2048 * 1024 * 1024 / per_item);
    if (const char *env = std::getenv("HECUDA_CHUNK")) chunk = std::atoll(env);
    h->chunk = std::max<int64_t>(1, std::min<int64_t>(chunk, 4096));
    context_registered(h, true);
    *out = h;
    return HECUDA_OK;
}

int32_t hecuda_context_destroy(hecuda_context *h) {
    if (!h) return HECUDA_OK;
    if (h->ctx) cudaSetDevice(h->ctx->device);
    cudaDeviceSynchronize();
    pir_graphs_purge(h, nullptr);
    context_registered(h, false);
    for (Workspace *w : h->free_ws) {
        w->release();
        delete w;
    }
    delete h->ctx;
    delete h;
    return HECUDA_OK;
}

int32_t hecuda_context_ciphertext_moduli_count(const hecuda_context *h, int32_t *count) {
    if (!h || !count) return fail(HECUDA_ERR_INVALID_ARGUMENT, "null argument");
    *count = h->ctx->L;
    return HECUDA_OK;
}
int32_t hecuda_context_bsk_moduli(const hecuda_context *h, uint64_t *out, int32_t capacity, int32_t *count) {
    if (!h || !count) return fail(HECUDA_ERR_INVALID_ARGUMENT, "null argument");
    *count = (int32_t)h->ctx->bsk.size();
    if (out) {
        if (capacity < *count) return fail(HECUDA_ERR_INVALID_ARGUMENT, "capacity too small");
        std::memcpy(out, h->ctx->bsk.data(), sizeof(u64) * h->ctx->bsk.size());
    }
    return HECUDA_OK;
}
int32_t hecuda_context_aux_moduli(const hecuda_context *h, uint64_t *out, int32_t capacity, int32_t *count) {
    if (!h || !count) return fail(HECUDA_ERR_INVALID_ARGUMENT, "null argument");
    *count = (int32_t)h->ctx->aux.size();
    if (out) {
        if (capacity < *count) return fail(HECUDA_ERR_INVALID_ARGUMENT, "capacity too small");
        std::memcpy(out, h->ctx->aux.data(), sizeof(u64) * h->ctx->aux.size());
    }
    return HECUDA_OK;
}
int32_t hecuda_context_root_tables(const hecuda_context *h, uint64_t modulus, uint64_t *roots, uint64_t *inverse_roots) {
    if (!h) return fail(HECUDA_ERR_INVALID_ARGUMENT, "null context");
    const int s = h->ctx->find_slot(modulus);
    if (s < 0) return fail(HECUDA_ERR_INVALID_ARGUMENT, "invalidNttModulus: modulus is not part of this context");
    if (roots) std::memcpy(roots, h->ctx->slots[s].roots.data(), sizeof(u64) * h->ctx->n);
    if (inverse_roots) std::memcpy(inverse_roots, h->ctx->slots[s].inv_roots.data(), sizeof(u64) * h->ctx->n);
    return HECUDA_OK;
}

// ---------------------------------------------------------------- NTT

// In place: `items` items of `rows_per_item` rows (`words_per_item` words) each.
static int32_t ntt_run(const hecuda_context *h, Io io, void *stream, const NttRowMap &map, void *data, size_t words_per_item,
                       int64_t items, int64_t rows_per_item, bool inverse) {
    const Context &c = *h->ctx;
    return dispatch(h, io, stream, "ntt launch", items, stage_items(words_per_item), 0, {{(const u64 *)data, words_per_item}},
                    data, words_per_item, [&](const Chunk &k) {
                        return inverse ? launch_ntt_inverse(c, map, k.in[0], k.out, k.items * rows_per_item, kScalePlain, k.stream)
                                       : launch_ntt_forward(c, map, k.in[0], k.out, k.items * rows_per_item, k.stream);
                    });
}
static int32_t ntt(const hecuda_context *h, int32_t base, void *data, int32_t rows, int64_t polys, bool inverse, Io io,
                   void *stream = nullptr) {
    int32_t rc = check_io(h, io);
    if (rc || (rc = check_batch(polys, {data}, "invalid data / poly_count"))) return rc;
    NttRowMap map;
    std::string err;
    if (!make_map(*h->ctx, base, rows, map, err)) return fail(HECUDA_ERR_INVALID_ARGUMENT, err);
    return ntt_run(h, io, stream, map, data, (size_t)rows * h->ctx->n, polys, rows, inverse);
}
int32_t hecuda_ntt_forward_device(const hecuda_context *h, int32_t base, uint64_t *data, int32_t rows, int64_t polys,
                                  void *stream) {
    return ntt(h, base, data, rows, polys, false, Io::Device, stream);
}
int32_t hecuda_ntt_inverse_device(const hecuda_context *h, int32_t base, uint64_t *data, int32_t rows, int64_t polys,
                                  void *stream) {
    return ntt(h, base, data, rows, polys, true, Io::Device, stream);
}
int32_t hecuda_ntt_forward(const hecuda_context *h, int32_t base, uint64_t *data, int32_t rows, int64_t polys) {
    return ntt(h, base, data, rows, polys, false, Io::Host64);
}
int32_t hecuda_ntt_inverse(const hecuda_context *h, int32_t base, uint64_t *data, int32_t rows, int64_t polys) {
    return ntt(h, base, data, rows, polys, true, Io::Host64);
}

// Stage-level BEHZ entry points over the reference's [Q, Bsk] (RnsTool.swift:324-331, 453-456), Coeff format.
static int32_t lift_q_to_qbsk(const hecuda_context *h, const void *polys, void *out, int64_t count, Io io) {
    int32_t rc = check_io(h, io);
    if (rc || (rc = check_batch(count, {polys, out}, "invalid buffers / poly_count"))) return rc;
    const Context &c = *h->ctx;
    const size_t in_words = (size_t)c.L * c.n, out_words = (size_t)(2 * c.L + 1) * c.n;
    return dispatch(h, io, nullptr, "liftQToQBsk", count, stage_items(out_words), 0, {{(const u64 *)polys, in_words}}, out,
                    out_words, [&](const Chunk &k) {
                        return launch_lift(c, k.in[0], 1, k.out, 1, 0, k.items, k.stream, /*reference_base=*/true);
                    });
}
static int32_t floor_qbsk_to_q(const hecuda_context *h, const void *polys, void *out, int64_t count, Io io) {
    int32_t rc = check_io(h, io);
    if (rc || (rc = check_batch(count, {polys, out}, "invalid buffers / poly_count"))) return rc;
    const Context &c = *h->ctx;
    const size_t in_words = (size_t)(2 * c.L + 1) * c.n, out_words = (size_t)c.L * c.n;
    return dispatch(h, io, nullptr, "floorQBskToQ", count, stage_items(in_words), 0, {{(const u64 *)polys, in_words}}, out,
                    out_words, [&](const Chunk &k) {
                        return launch_floor(c, k.in[0], k.out, k.items, k.stream, /*reference_base=*/true);
                    });
}
int32_t hecuda_rnstool_lift_q_to_qbsk(const hecuda_context *h, const uint64_t *polys, uint64_t *out, int64_t count) {
    return lift_q_to_qbsk(h, polys, out, count, Io::Host64);
}
int32_t hecuda_rnstool_floor_qbsk_to_q(const hecuda_context *h, const uint64_t *polys, uint64_t *out, int64_t count) {
    return floor_qbsk_to_q(h, polys, out, count, Io::Host64);
}

static int32_t ntt_rows(const hecuda_context *h, uint64_t modulus, uint64_t *data, int64_t rows, bool inverse) {
    int32_t rc = check_ctx(h);
    if (rc || (rc = check_batch(rows, {data}, "invalid data / row_count"))) return rc;
    const int s = h->ctx->find_slot(modulus);
    if (s < 0) return fail(HECUDA_ERR_INVALID_ARGUMENT, "invalidPolyContext: modulus is not part of this context");
    return ntt_run(h, Io::Host64, nullptr, h->ctx->map_single(s), data, (size_t)h->ctx->n, rows, 1, inverse);
}
int32_t hecuda_ntt_forward_rows(const hecuda_context *h, uint64_t modulus, uint64_t *data, int64_t rows) {
    return ntt_rows(h, modulus, data, rows, false);
}
int32_t hecuda_ntt_inverse_rows(const hecuda_context *h, uint64_t modulus, uint64_t *data, int64_t rows) {
    return ntt_rows(h, modulus, data, rows, true);
}

// ---------------------------------------------------------------- multiply

static int32_t multiply(const hecuda_context *h, const void *lhs, const void *rhs, void *out, int64_t batch, Io io,
                        void *stream = nullptr) {
    int32_t rc = check_io(h, io);
    if (rc || (rc = check_batch(batch, {lhs, rhs, out}, "invalidCiphertext: null buffer"))) return rc;
    const Context &c = *h->ctx;
    const size_t in_words = (size_t)2 * c.L * c.n, out_words = (size_t)3 * c.L * c.n;
    return dispatch(h, io, stream, "multiply", batch, h->chunk, multiply_scratch_words(c),
                    {{(const u64 *)lhs, in_words}, {(const u64 *)rhs, in_words}}, out, out_words, [&](const Chunk &k) {
                        return multiply_chunk(c, k.scratch, k.in[0], k.in[1], k.out, k.items, k.stream);
                    });
}
int32_t hecuda_bfv_multiply_device(const hecuda_context *h, const uint64_t *lhs, const uint64_t *rhs, uint64_t *out,
                                   int64_t batch, void *stream) {
    return multiply(h, lhs, rhs, out, batch, Io::Device, stream);
}
int32_t hecuda_bfv_multiply(const hecuda_context *h, const uint64_t *lhs, const uint64_t *rhs, uint64_t *out,
                            int64_t batch) {
    return multiply(h, lhs, rhs, out, batch, Io::Host64);
}

// ---------------------------------------------------------------- evaluation key

int32_t hecuda_evk_create_empty(const hecuda_context *h, hecuda_evk **out) {
    int32_t rc = check_ctx(h);
    if (rc) return rc;
    if (!out) return fail(HECUDA_ERR_INVALID_ARGUMENT, "null argument");
    const Context &c = *h->ctx;
    if (!c.has_ks)  // Context.supportsEvaluationKey == false with a single coefficient modulus (Context.swift:102-107)
        return fail(HECUDA_ERR_UNSUPPORTED, "unsupportedHeOperation: a single coefficient modulus leaves no key-switching modulus");
    hecuda_evk *k = new (std::nothrow) hecuda_evk();
    if (!k) return fail(HECUDA_ERR_CUDA, "out of host memory");
    k->owner = h;
    k->words = (size_t)c.L * 2 * (c.L + 1) * c.n;
    cudaError_t e = cudaMalloc(&k->d_relin, k->words * sizeof(u64));
    if (e != cudaSuccess) {
        delete k;
        return cuda_fail(e, "cudaMalloc(evk)");
    }
    *out = k;
    return HECUDA_OK;
}
int32_t hecuda_evk_create(const hecuda_context *h, const uint64_t *relin_key, hecuda_evk **out) {
    if (!relin_key) return fail(HECUDA_ERR_MISSING_KEY, "missingRelinearizationKey");
    int32_t rc = hecuda_evk_create_empty(h, out);
    if (rc) return rc;
    cudaError_t e = upload((*out)->d_relin, relin_key, (*out)->words * sizeof(u64));
    if (e != cudaSuccess) {
        hecuda_evk_destroy(*out);
        *out = nullptr;
        return cuda_fail(e, "cudaMemcpy(evk)");
    }
    (*out)->loaded = true;
    return HECUDA_OK;
}
int32_t hecuda_evk_destroy(hecuda_evk *k) {
    if (!k) return HECUDA_OK;
    if (k->owner) pir_graphs_purge(const_cast<hecuda_context *>(k->owner), k);
    if (k->d_relin) cudaFree(k->d_relin);
    for (auto &kv : k->galois) cudaFree(kv.second);
    for (hecuda::u64 *p : k->retired) cudaFree(p);
    delete k;
    return HECUDA_OK;
}
int32_t hecuda_evk_device_buffer(hecuda_evk *k, void **device_ptr, uint64_t *bytes) {
    if (!k || !device_ptr || !bytes) return fail(HECUDA_ERR_INVALID_ARGUMENT, "null argument");
    *device_ptr = k->d_relin;
    *bytes = k->words * sizeof(u64);
    k->loaded = true;  // the caller fills it (e.g. ncclBroadcast from rank 0)
    ++k->version;
    return HECUDA_OK;
}

// ---------------------------------------------------------------- relinearize / mod switch

static int32_t relinearize(const hecuda_context *h, const hecuda_evk *k, const void *ct3, int32_t l, void *out,
                           int64_t batch, Io io, void *stream = nullptr) {
    int32_t rc = check_io(h, io);
    if (rc || (rc = check_key(h, k, true)) || (rc = check_level(h, l, "invalidCiphertext")) ||
        (rc = check_batch(batch, {ct3, out}, "invalidCiphertext: null buffer")))
        return rc;
    const Context &c = *h->ctx;
    return dispatch(h, io, stream, "relinearize", batch, h->chunk, relinearize_scratch_words(c, l),
                    {{(const u64 *)ct3, (size_t)3 * l * c.n}}, out, (size_t)2 * l * c.n, [&](const Chunk &ch) {
                        return relinearize_chunk(c, ch.scratch, k->d_relin, ch.in[0], l, ch.out, ch.items, ch.stream);
                    });
}
int32_t hecuda_bfv_relinearize_device(const hecuda_context *h, const hecuda_evk *k, const uint64_t *ct3, int32_t l,
                                      uint64_t *out, int64_t batch, void *stream) {
    return relinearize(h, k, ct3, l, out, batch, Io::Device, stream);
}
int32_t hecuda_bfv_relinearize(const hecuda_context *h, const hecuda_evk *k, const uint64_t *ct3, int32_t l,
                               uint64_t *out, int64_t batch) {
    return relinearize(h, k, ct3, l, out, batch, Io::Host64);
}

static int32_t mod_switch_down(const hecuda_context *h, const void *ct, int32_t polys, int32_t l, void *out, int64_t batch,
                               Io io, void *stream = nullptr) {
    int32_t rc = check_io(h, io);
    if (rc) return rc;
    if (polys < 1) return fail(HECUDA_ERR_INVALID_ARGUMENT, "invalidCiphertext: poly_count");
    if (l < 2 || l > h->ctx->L)
        return fail(HECUDA_ERR_INVALID_ARGUMENT, "invalidPolyContext: modSwitchDown needs a next context (2 <= moduli_count <= L)");
    if ((rc = check_batch(batch, {ct, out}, "invalidCiphertext: null buffer"))) return rc;
    const Context &c = *h->ctx;
    const size_t in_words = (size_t)polys * l * c.n;
    return dispatch(h, io, stream, "mod_switch", batch, stage_items(in_words), 0, {{(const u64 *)ct, in_words}}, out,
                    (size_t)polys * (l - 1) * c.n, [&](const Chunk &k) {
                        return launch_mod_switch(c, k.in[0], l, k.out, k.items * polys, k.stream);
                    });
}
int32_t hecuda_bfv_mod_switch_down_device(const hecuda_context *h, const uint64_t *ct, int32_t polys, int32_t l,
                                          uint64_t *out, int64_t batch, void *stream) {
    return mod_switch_down(h, ct, polys, l, out, batch, Io::Device, stream);
}
int32_t hecuda_bfv_mod_switch_down(const hecuda_context *h, const uint64_t *ct, int32_t polys, int32_t l, uint64_t *out,
                                   int64_t batch) {
    return mod_switch_down(h, ct, polys, l, out, batch, Io::Host64);
}

// ---------------------------------------------------------------- relinearize -> modSwitchDown, fused
// Bfv.relinearize then Bfv.modSwitchDown on a batch in one pass (BASELINE config 3): the relinearized ciphertext stays
// in HBM, 2 x (l-1) rows per ciphertext come back.
static int32_t relinearize_mod_switch_down(const hecuda_context *h, const hecuda_evk *k, const void *ct3, int32_t l,
                                           void *out, int64_t batch, Io io) {
    int32_t rc = check_io(h, io);
    if (rc || (rc = check_key(h, k, true)) || (rc = check_level(h, l, "invalidCiphertext")) ||
        (rc = check_batch(batch, {ct3, out}, "invalidCiphertext: null buffer")))
        return rc;
    if (l < 2) return fail(HECUDA_ERR_INVALID_ARGUMENT, "invalidPolyContext: modSwitchDown needs a next context (moduli_count >= 2)");
    const Context &c = *h->ctx;
    const size_t relin_words = (size_t)2 * l * c.n;
    return dispatch(h, io, nullptr, "relinearize_mod_switch_down", batch, h->chunk,
                    relinearize_scratch_words(c, l) + relin_words, {{(const u64 *)ct3, (size_t)3 * l * c.n}}, out,
                    (size_t)2 * (l - 1) * c.n, [&](const Chunk &ch) {
                        u64 *relin = ch.scratch + relinearize_scratch_words(c, l) * (size_t)ch.items;
                        cudaError_t e = relinearize_chunk(c, ch.scratch, k->d_relin, ch.in[0], l, relin, ch.items, ch.stream);
                        if (e != cudaSuccess) return e;
                        return launch_mod_switch(c, relin, l, ch.out, ch.items * 2, ch.stream);
                    });
}
int32_t hecuda_bfv_relinearize_mod_switch_down(const hecuda_context *h, const hecuda_evk *k, const uint64_t *ct3, int32_t l,
                                               uint64_t *out, int64_t batch) {
    return relinearize_mod_switch_down(h, k, ct3, l, out, batch, Io::Host64);
}

// ---------------------------------------------------------------- multiply -> relinearize (-> modSwitchDown), fused
// The sequence every caller of ct x ct multiply runs (RlweBenchmark.swift:387-493; PirUtil.swift:447-480):
// Bfv.mulAssign, Bfv.relinearize, optionally Bfv.modSwitchDown, on a batch, in one pass: the three-polynomial product
// and the relinearized ciphertext stay in HBM and only 2 x L (or 2 x (L-1)) rows per ciphertext come back.
static size_t mul_relin_scratch_words(const Context &c) {
    // multiply scratch | 3-poly product | relinearize scratch | relinearized ciphertext (only with the modulus switch)
    return multiply_scratch_words(c) + (size_t)3 * c.L * c.n + relinearize_scratch_words(c, c.L) + (size_t)2 * c.L * c.n;
}
static cudaError_t mul_relin_chunk(const Context &c, u64 *scratch, const u64 *key, const u64 *lhs, const u64 *rhs, bool mod_switch,
                                   u64 *out, int64_t items, cudaStream_t s) {
    u64 *mul_scratch = scratch;
    u64 *prod = mul_scratch + multiply_scratch_words(c) * (size_t)items;
    u64 *ks_scratch = prod + (size_t)3 * c.L * c.n * items;
    u64 *relin = ks_scratch + relinearize_scratch_words(c, c.L) * (size_t)items;
    cudaError_t e;
    if ((e = multiply_chunk(c, mul_scratch, lhs, rhs, prod, items, s)) != cudaSuccess) return e;
    if ((e = relinearize_chunk(c, ks_scratch, key, prod, c.L, mod_switch ? relin : out, items, s)) != cudaSuccess) return e;
    if (mod_switch) return launch_mod_switch(c, relin, c.L, out, items * 2, s);
    return cudaSuccess;
}
static int32_t multiply_relinearize(const hecuda_context *h, const hecuda_evk *k, const void *lhs, const void *rhs,
                                    int32_t mod_switch, void *out, int64_t batch, Io io, void *stream = nullptr) {
    int32_t rc = check_io(h, io);
    if (rc || (rc = check_key(h, k, true))) return rc;
    if (mod_switch && h->ctx->L < 2)
        return fail(HECUDA_ERR_INVALID_ARGUMENT, "invalidPolyContext: modSwitchDown needs a next context (L >= 2)");
    if ((rc = check_batch(batch, {lhs, rhs, out}, "invalidCiphertext: null buffer"))) return rc;
    const Context &c = *h->ctx;
    const size_t in_words = (size_t)2 * c.L * c.n, out_words = (size_t)2 * (c.L - (mod_switch ? 1 : 0)) * c.n;
    return dispatch(h, io, stream, "multiply_relinearize", batch, std::max<int64_t>(1, h->chunk / 2),
                    mul_relin_scratch_words(c), {{(const u64 *)lhs, in_words}, {(const u64 *)rhs, in_words}}, out, out_words,
                    [&](const Chunk &ch) {
                        return mul_relin_chunk(c, ch.scratch, k->d_relin, ch.in[0], ch.in[1], mod_switch != 0, ch.out,
                                               ch.items, ch.stream);
                    });
}
int32_t hecuda_bfv_multiply_relinearize_device(const hecuda_context *h, const hecuda_evk *k, const uint64_t *lhs,
                                               const uint64_t *rhs, int32_t mod_switch, uint64_t *out, int64_t batch,
                                               void *stream) {
    return multiply_relinearize(h, k, lhs, rhs, mod_switch, out, batch, Io::Device, stream);
}
int32_t hecuda_bfv_multiply_relinearize(const hecuda_context *h, const hecuda_evk *k, const uint64_t *lhs, const uint64_t *rhs,
                                        int32_t mod_switch, uint64_t *out, int64_t batch) {
    return multiply_relinearize(h, k, lhs, rhs, mod_switch, out, batch, Io::Host64);
}

// ---------------------------------------------------------------- Galois (SURVEY.md 8f rank 1)

static bool valid_galois_element(int64_t element, int64_t n) {  // isValidGaloisElement, Galois.swift:100-105
    return (element & 1) && element > 1 && element < 2 * n;
}

int32_t hecuda_evk_set_galois_key(hecuda_evk *k, uint32_t element, const uint64_t *key) {
    if (!k || !key) return fail(HECUDA_ERR_INVALID_ARGUMENT, "null argument");
    int32_t rc = check_ctx(k->owner);
    if (rc) return rc;
    if (!valid_galois_element(element, k->owner->ctx->n)) return fail(HECUDA_ERR_INVALID_ARGUMENT, "invalid Galois element");
    u64 *d = nullptr;
    CK(cudaMalloc(&d, k->words * sizeof(u64)));
    cudaError_t e = upload(d, key, k->words * sizeof(u64));
    if (e != cudaSuccess) {
        cudaFree(d);
        return cuda_fail(e, "cudaMemcpy(galois key)");
    }
    std::lock_guard<std::mutex> g(k->mu);
    auto it = k->galois.find(element);
    if (it != k->galois.end()) {
        // kernels already enqueued by other threads may still read the key being replaced (callers copy the device
        // pointer out under the mutex and launch afterwards): retire the buffer, free it with the handle
        k->retired.push_back(it->second);
        it->second = d;
    } else {
        k->galois[element] = d;
    }
    ++k->version;  // captured pipelines (pir.cu) bake the key pointers in: they are rebuilt on the next call
    return HECUDA_OK;
}

int32_t hecuda_evk_galois_device_buffer(hecuda_evk *k, uint32_t element, void **device_ptr, uint64_t *bytes) {
    if (!k || !device_ptr || !bytes) return fail(HECUDA_ERR_INVALID_ARGUMENT, "null argument");
    int32_t rc = check_ctx(k->owner);
    if (rc) return rc;
    if (!valid_galois_element(element, k->owner->ctx->n)) return fail(HECUDA_ERR_INVALID_ARGUMENT, "invalid Galois element");
    std::lock_guard<std::mutex> g(k->mu);
    auto it = k->galois.find(element);
    if (it == k->galois.end()) {  // the caller fills it (e.g. ncclBroadcast from the rank that holds the key)
        u64 *d = nullptr;
        CK(cudaMalloc(&d, k->words * sizeof(u64)));
        it = k->galois.emplace(element, d).first;
    }
    *device_ptr = it->second;
    *bytes = k->words * sizeof(u64);
    return HECUDA_OK;
}

static int32_t apply_galois(const hecuda_context *h, const hecuda_evk *k, const void *ct, int32_t l, uint32_t element,
                            void *out, int64_t batch, Io io, void *stream = nullptr) {
    int32_t rc = check_io(h, io);
    if (rc || (rc = check_key(h, k, false))) return rc;
    if (!valid_galois_element(element, h->ctx->n)) return fail(HECUDA_ERR_INVALID_ARGUMENT, "invalid Galois element");
    if ((rc = check_level(h, l, "invalidCiphertext")) || (rc = check_batch(batch, {ct, out}, "invalidCiphertext: null buffer")))
        return rc;
    const u64 *key = nullptr;
    {
        hecuda_evk *km = const_cast<hecuda_evk *>(k);
        std::lock_guard<std::mutex> g(km->mu);
        auto it = km->galois.find(element);
        if (it == km->galois.end()) return fail(HECUDA_ERR_MISSING_KEY, "missingGaloisElement: " + std::to_string(element));
        key = it->second;
    }
    const Context &c = *h->ctx;
    const size_t words = (size_t)2 * l * c.n;
    return dispatch(h, io, stream, "applyGalois", batch, h->chunk, galois_scratch_words(c, l), {{(const u64 *)ct, words}},
                    out, words, [&](const Chunk &ch) {
                        return apply_galois_chunk(c, ch.scratch, key, ch.in[0], l, element, ch.out, ch.items, ch.stream);
                    });
}
int32_t hecuda_bfv_apply_galois_device(const hecuda_context *h, const hecuda_evk *k, const uint64_t *ct, int32_t l,
                                       uint32_t element, uint64_t *out, int64_t batch, void *stream) {
    return apply_galois(h, k, ct, l, element, out, batch, Io::Device, stream);
}
int32_t hecuda_bfv_apply_galois(const hecuda_context *h, const hecuda_evk *k, const uint64_t *ct, int32_t l,
                                uint32_t element, uint64_t *out, int64_t batch) {
    return apply_galois(h, k, ct, l, element, out, batch, Io::Host64);
}

int32_t hecuda_poly_apply_galois(const hecuda_context *h, int32_t base, int32_t eval_format, const uint64_t *in,
                                 uint64_t *out, int32_t rows, int64_t polys, uint32_t element) {
    int32_t rc = check_ctx(h);
    if (rc || (rc = check_batch(polys, {in, out}, "invalid data / poly_count"))) return rc;
    if (!valid_galois_element(element, h->ctx->n)) return fail(HECUDA_ERR_INVALID_ARGUMENT, "invalid Galois element");
    NttRowMap map;
    std::string err;
    if (!make_map(*h->ctx, base, rows, map, err)) return fail(HECUDA_ERR_INVALID_ARGUMENT, err);
    const Context &c = *h->ctx;
    const size_t words = (size_t)rows * c.n;
    return dispatch(h, Io::Host64, nullptr, "poly_apply_galois", polys, stage_items(words), 0, {{(const u64 *)in, words}}, out,
                    words, [&](const Chunk &k) {
                        return eval_format ? launch_galois_eval(c, rows, element, k.in[0], k.out, k.items, k.stream)
                                           : launch_galois_coeff(c, map, element, k.in[0], (int64_t)words, k.out,
                                                                 (int64_t)words, k.items, k.stream);
                    });
}

// ---------------------------------------------------------------- lazy ct x pt inner product (SURVEY.md 8f rank 2)

static int32_t inner_product_plaintexts(const hecuda_context *h, const void *cts, int32_t polys, int32_t l, int64_t terms,
                                        const void *pts, const uint8_t *present, void *out, int64_t out_count, Io io,
                                        void *stream = nullptr) {
    int32_t rc = check_io(h, io);
    if (rc) return rc;
    if (polys < 1 || polys > 3) return fail(HECUDA_ERR_INVALID_ARGUMENT, "invalidCiphertext: poly_count must be 1..3");
    if ((rc = check_level(h, l, "invalidCiphertext"))) return rc;
    if (terms < 1) return fail(HECUDA_ERR_INVALID_ARGUMENT, "Empty ciphertexts");  // precondition, Bfv.swift:481-483
    if ((rc = check_batch(out_count, {cts, pts, out}, "null buffer"))) return rc;
    if (h->ctx->n < 2) return fail(HECUDA_ERR_UNSUPPORTED, "degree too small");
    if (out_count == 0) return HECUDA_OK;
    const Context &c = *h->ctx;
    // the query ciphertexts (and the presence flags) are shared by every output row: a host call uploads them once
    u64 *d_cts = nullptr;
    unsigned char *d_present = nullptr;
    if (io == Io::Host64) {
        const size_t ct_words = (size_t)terms * polys * l * c.n;
        CK(cudaMalloc(&d_cts, ct_words * sizeof(u64)));
        cudaError_t e = upload(d_cts, cts, ct_words * sizeof(u64));
        if (e == cudaSuccess && present) {
            e = cudaMalloc(&d_present, (size_t)out_count * terms);
            if (e == cudaSuccess) e = upload(d_present, present, (size_t)out_count * terms);
        }
        if (e != cudaSuccess) {
            cudaFree(d_cts);
            cudaFree(d_present);
            return cuda_fail(e, "inner_product upload");
        }
        cts = d_cts;
        present = d_present;
    }
    const size_t pt_words = (size_t)terms * l * c.n;
    rc = dispatch(h, io, stream, "inner_product", out_count, stage_items(pt_words, (size_t)32 * 1024 * 1024),
                  0, {{(const u64 *)pts, pt_words}}, out, (size_t)polys * l * c.n, [&](const Chunk &k) {
                      const unsigned char *pr = present ? present + k.first * terms : nullptr;
                      return launch_inner_product_plain(c, (const u64 *)cts, polys, l, terms, k.in[0], pr, k.out, k.items, k.stream);
                  });
    if (io == Io::Host64) {
        cudaDeviceSynchronize();
        cudaFree(d_cts);
        cudaFree(d_present);
    }
    return rc;
}
int32_t hecuda_bfv_inner_product_plaintexts_device(const hecuda_context *h, const uint64_t *cts, int32_t polys,
                                                   int32_t l, int64_t terms, const uint64_t *pts,
                                                   const uint8_t *present, uint64_t *out, int64_t out_count,
                                                   void *stream) {
    return inner_product_plaintexts(h, cts, polys, l, terms, pts, present, out, out_count, Io::Device, stream);
}
int32_t hecuda_bfv_inner_product_plaintexts(const hecuda_context *h, const uint64_t *cts, int32_t polys, int32_t l,
                                            int64_t terms, const uint64_t *pts, const uint8_t *present, uint64_t *out,
                                            int64_t out_count) {
    return inner_product_plaintexts(h, cts, polys, l, terms, pts, present, out, out_count, Io::Host64);
}

static int32_t plaintext_to_eval(const hecuda_context *h, const void *plain, int32_t l, void *out, int64_t count, Io io,
                                 void *stream = nullptr) {
    int32_t rc = check_io(h, io);
    if (rc || (rc = check_level(h, l, "invalidPolyContext")) || (rc = check_batch(count, {plain, out}, "null buffer")))
        return rc;
    const Context &c = *h->ctx;
    return dispatch(h, io, stream, "plaintext_to_eval", count, stage_items((size_t)l * c.n), 0, {{(const u64 *)plain, (size_t)c.n}}, out,
                    (size_t)l * c.n, [&](const Chunk &k) {
                        return launch_plaintext_to_eval(c, k.in[0], l, k.out, k.items, k.stream);
                    });
}
int32_t hecuda_plaintext_to_eval_device(const hecuda_context *h, const uint64_t *plain, int32_t l, uint64_t *out,
                                        int64_t count, void *stream) {
    return plaintext_to_eval(h, plain, l, out, count, Io::Device, stream);
}
int32_t hecuda_plaintext_to_eval(const hecuda_context *h, const uint64_t *plain, int32_t l, uint64_t *out,
                                 int64_t count) {
    return plaintext_to_eval(h, plain, l, out, count, Io::Host64);
}

// ---------------------------------------------------------------- ct x ct inner product (SURVEY.md 8f rank 2)

static int32_t inner_product(const hecuda_context *h, const void *lhs, const void *rhs, void *out, int64_t pairs,
                             int64_t groups, Io io, void *stream = nullptr) {
    int32_t rc = check_io(h, io);
    if (rc) return rc;
    if (pairs < 1) return fail(HECUDA_ERR_INVALID_ARGUMENT, "Empty ciphertexts");
    if ((rc = check_batch(groups, {lhs, rhs, out}, "invalidCiphertext: null buffer"))) return rc;
    if (h->ctx->n < 2) return fail(HECUDA_ERR_UNSUPPORTED, "degree too small");
    const Context &c = *h->ctx;
    const size_t in_words = (size_t)pairs * 2 * c.L * c.n;
    return dispatch(h, io, stream, "innerProduct", groups, std::max<int64_t>(1, h->chunk / pairs),
                    inner_product_scratch_words(c, pairs), {{(const u64 *)lhs, in_words}, {(const u64 *)rhs, in_words}},
                    out, (size_t)3 * c.L * c.n, [&](const Chunk &k) {
                        return inner_product_chunk(c, k.scratch, k.in[0], k.in[1], pairs, k.out, k.items, k.stream);
                    });
}
int32_t hecuda_bfv_inner_product_device(const hecuda_context *h, const uint64_t *lhs, const uint64_t *rhs, uint64_t *out,
                                        int64_t pairs, int64_t groups, void *stream) {
    return inner_product(h, lhs, rhs, out, pairs, groups, Io::Device, stream);
}
int32_t hecuda_bfv_inner_product(const hecuda_context *h, const uint64_t *lhs, const uint64_t *rhs, uint64_t *out,
                                 int64_t pairs, int64_t groups) {
    return inner_product(h, lhs, rhs, out, pairs, groups, Io::Host64);
}

int32_t hecuda_poly_multiply_power_of_x(const hecuda_context *h, int32_t base, const uint64_t *in, uint64_t *out,
                                        int32_t rows, int64_t polys, int64_t power) {
    int32_t rc = check_ctx(h);
    if (rc || (rc = check_batch(polys, {in, out}, "invalid data / poly_count"))) return rc;
    NttRowMap map;
    std::string err;
    if (!make_map(*h->ctx, base, rows, map, err)) return fail(HECUDA_ERR_INVALID_ARGUMENT, err);
    const Context &c = *h->ctx;
    const size_t words = (size_t)rows * c.n;
    return dispatch(h, Io::Host64, nullptr, "multiply_power_of_x", polys, stage_items(words), 0, {{(const u64 *)in, words}}, out, words,
                    [&](const Chunk &k) {
                        return launch_multiply_power_of_x(c, map, power, k.in[0], k.out, k.items, k.stream);
                    });
}

uint64_t hecuda_kernel_launch_count(void) { return g_kernel_launches.load(); }


// ---------------------------------------------------------------- Bfv<UInt32>: uint32 buffers at the boundary
// (the reference's second scalar type, HeScheme.swift / Scalar.swift:498-511).  Same layouts as the uint64 entry points;
// the context must have been made by hecuda_context_create_u32 (its m~, gamma and Bsk).
int32_t hecuda_u32_ntt_forward(const hecuda_context *h, int32_t base, uint32_t *data, int32_t rows, int64_t polys) {
    return ntt(h, base, data, rows, polys, false, Io::Host32);
}
int32_t hecuda_u32_ntt_inverse(const hecuda_context *h, int32_t base, uint32_t *data, int32_t rows, int64_t polys) {
    return ntt(h, base, data, rows, polys, true, Io::Host32);
}
int32_t hecuda_u32_bfv_multiply(const hecuda_context *h, const uint32_t *lhs, const uint32_t *rhs, uint32_t *out, int64_t batch) {
    return multiply(h, lhs, rhs, out, batch, Io::Host32);
}
int32_t hecuda_u32_evk_create(const hecuda_context *h, const uint32_t *relin_key, hecuda_evk **out) {
    int32_t rc = need_word32(h);
    if (rc) return rc;
    if (!relin_key) return fail(HECUDA_ERR_MISSING_KEY, "missingRelinearizationKey");
    const Context &c = *h->ctx;
    const size_t words = (size_t)c.L * 2 * (c.L + 1) * c.n;
    std::vector<uint64_t> wide(relin_key, relin_key + words);  // setup-time: widened on the host
    return hecuda_evk_create(h, wide.data(), out);
}
int32_t hecuda_u32_bfv_relinearize(const hecuda_context *h, const hecuda_evk *evk, const uint32_t *ct3, int32_t l, uint32_t *out,
                                   int64_t batch) {
    return relinearize(h, evk, ct3, l, out, batch, Io::Host32);
}
int32_t hecuda_u32_bfv_mod_switch_down(const hecuda_context *h, const uint32_t *ct, int32_t polys, int32_t l, uint32_t *out,
                                       int64_t batch) {
    return mod_switch_down(h, ct, polys, l, out, batch, Io::Host32);
}
int32_t hecuda_u32_bfv_multiply_relinearize(const hecuda_context *h, const hecuda_evk *evk, const uint32_t *lhs, const uint32_t *rhs,
                                            int32_t mod_switch, uint32_t *out, int64_t batch) {
    return multiply_relinearize(h, evk, lhs, rhs, mod_switch, out, batch, Io::Host32);
}
int32_t hecuda_u32_bfv_relinearize_mod_switch_down(const hecuda_context *h, const hecuda_evk *evk, const uint32_t *ct3, int32_t l,
                                                   uint32_t *out, int64_t batch) {
    return relinearize_mod_switch_down(h, evk, ct3, l, out, batch, Io::Host32);
}
int32_t hecuda_u32_evk_set_galois_key(hecuda_evk *evk, uint32_t element, const uint32_t *key) {
    if (!evk || !key) return fail(HECUDA_ERR_INVALID_ARGUMENT, "null argument");
    int32_t rc = need_word32(evk->owner);
    if (rc) return rc;
    std::vector<uint64_t> wide(key, key + evk->words);  // setup-time: widened on the host
    return hecuda_evk_set_galois_key(evk, element, wide.data());
}
int32_t hecuda_u32_bfv_apply_galois(const hecuda_context *h, const hecuda_evk *evk, const uint32_t *ct, int32_t l, uint32_t element,
                                    uint32_t *out, int64_t batch) {
    return apply_galois(h, evk, ct, l, element, out, batch, Io::Host32);
}
int32_t hecuda_u32_bfv_inner_product(const hecuda_context *h, const uint32_t *lhs, const uint32_t *rhs, uint32_t *out, int64_t pairs,
                                     int64_t groups) {
    return inner_product(h, lhs, rhs, out, pairs, groups, Io::Host32);
}
int32_t hecuda_u32_rnstool_lift_q_to_qbsk(const hecuda_context *h, const uint32_t *polys, uint32_t *out, int64_t count) {
    return lift_q_to_qbsk(h, polys, out, count, Io::Host32);
}
int32_t hecuda_u32_rnstool_floor_qbsk_to_q(const hecuda_context *h, const uint32_t *polys, uint32_t *out, int64_t count) {
    return floor_qbsk_to_q(h, polys, out, count, Io::Host32);
}

}  // extern "C"
