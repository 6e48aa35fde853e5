// C ABI (include/snark_setup_b200.h) and the host-side driver of the batch-exponentiation path.
//
// Host logic mirrors, in C++, the orchestration the reference keeps in Rust:
//   Phase1Parameters::new / chunk_sizes   phase1/src/objects/parameters.rs:115-294
//   split / split_mut                     phase1/src/helpers/buffers.rs:246-341
//   apply_powers                          phase1/src/helpers/buffers.rs:77-97
//   Phase1::computation                   phase1/src/computation.rs:40-302
// The reference walks each vector in `batch_size` windows on rayon threads; results do not depend
// on the windowing, so here each vector is cut into device tiles (default 1 212 416 elements) that are
// pipelined over two CUDA streams (H2D of tile k+1 overlaps the kernels of tile k), the five vectors
// of a call run on concurrent lanes, and with several devices every vector is split D ways.
#ifndef __CUDACC__
#error "api.cu is the CUDA product path and must be built with nvcc (no CPU fallback exists)"
#endif
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/snark_setup_b200.h"
#include "fft.cuh"
#include "msm.cuh"
#include "pairing.cuh"
#include "qap.cuh"

namespace {

using namespace ss;

thread_local ss_error_info g_err = {0, 0, 0, 0, {0}};

int fail(int code, uint64_t index, uint64_t expected, uint64_t got, const char* fmt, ...) {
    g_err.code = code;
    g_err.index = index;
    g_err.expected = expected;
    g_err.got = got;
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err.message, sizeof(g_err.message), fmt, ap);
    va_end(ap);
    return code;
}

#define CU(expr)                                                                                       \
    do {                                                                                               \
        cudaError_t _e = (expr);                                                                       \
        if (_e != cudaSuccess)                                                                         \
            return fail(SS_ERR_DEVICE, 0, 0, 0, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                        __FILE__, __LINE__);                                                           \
    } while (0)

const GroupOps* group_ops(int curve, int group) {
    if (curve == SS_CURVE_BLS12_377) return group == SS_G1 ? &ops_bls377_g1() : group == SS_G2 ? &ops_bls377_g2() : nullptr;
    if (curve == SS_CURVE_BW6_761) return group == SS_G1 ? &ops_bw6_g1() : group == SS_G2 ? &ops_bw6_g2() : nullptr;
    if (curve == SS_CURVE_MNT4_753) return group == SS_G1 ? &ops_mnt4_g1() : group == SS_G2 ? &ops_mnt4_g2() : nullptr;
    if (curve == SS_CURVE_MNT6_753) return group == SS_G1 ? &ops_mnt6_g1() : group == SS_G2 ? &ops_mnt6_g2() : nullptr;
    return nullptr;
}

// Scalars cross the ABI as ceil(bits / 8) canonical bytes (95 for the MNT curves); on the device every scalar occupies
// fr_words whole words.  Arrays of host scalars whose size is not a multiple of 4 are re-packed to that stride before
// the upload (`keep` owns the staging copy until the stream has been synchronised).
size_t scalar_stride(const GroupOps& o) { return (size_t)o.fr_words * 4; }
const uint8_t* repack_scalars(const GroupOps& o, const uint8_t* src, size_t n, std::vector<std::vector<uint8_t>>& keep) {
    const size_t fb = o.fr_bytes, fs = scalar_stride(o);
    if (fb == fs) return src;
    keep.emplace_back(n * fs, 0);
    uint8_t* dst = keep.back().data();
    for (size_t i = 0; i < n; i++) memcpy(dst + i * fs, src + i * fb, fb);
    return dst;
}

// ---- per-kernel timing (ss_profile_*) -----------------------------------------------------------
// When enabled every launch is bracketed by two CUDA events recorded on the launching stream; the
// pairs are resolved after the stream has been synchronised.  bench.py uses this for the per-kernel
// durations behind `roofline` and for `gpu_launches`.
std::mutex g_prof_mu;
bool g_prof_on = false;
struct ProfAcc {
    std::string name;
    uint64_t launches = 0, elements = 0;
    double ms = 0;
};
std::vector<ProfAcc> g_prof;
struct ProfPending {
    std::string name;
    uint64_t elements;
    cudaEvent_t e0, e1;
};
thread_local std::vector<ProfPending> g_prof_pending;
std::atomic<uint64_t> g_launches{0};

struct ProfScope {
    bool on;
    ProfPending p;
    cudaStream_t s;
    ProfScope(const char* kind, const char* group, uint64_t elements, cudaStream_t stream) : s(stream) {
        g_launches.fetch_add(1, std::memory_order_relaxed);
        on = g_prof_on;
        if (!on) return;
        p.name = std::string(kind) + "<" + group + ">";
        p.elements = elements;
        cudaEventCreate(&p.e0);
        cudaEventCreate(&p.e1);
        cudaEventRecord(p.e0, s);
    }
    ~ProfScope() {
        if (!on) return;
        cudaEventRecord(p.e1, s);
        g_prof_pending.push_back(p);
    }
};

// call after the streams used since the last flush have been synchronised
void prof_flush() {
    if (g_prof_pending.empty()) return;
    std::lock_guard<std::mutex> lk(g_prof_mu);
    for (auto& p : g_prof_pending) {
        float ms = 0;
        if (cudaEventSynchronize(p.e1) == cudaSuccess) cudaEventElapsedTime(&ms, p.e0, p.e1);
        cudaEventDestroy(p.e0);
        cudaEventDestroy(p.e1);
        ProfAcc* a = nullptr;
        for (auto& x : g_prof)
            if (x.name == p.name) a = &x;
        if (!a) {
            g_prof.push_back(ProfAcc());
            a = &g_prof.back();
            a->name = p.name;
        }
        a->launches++;
        a->elements += p.elements;
        a->ms += ms;
    }
    g_prof_pending.clear();
}

// ---- devices ------------------------------------------------------------------------------------
std::mutex g_mu;
std::vector<int> g_devices;
bool g_inited = false;

int ensure_init() {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_inited) return SS_OK;
    int cnt = 0;
    cudaError_t e = cudaGetDeviceCount(&cnt);
    if (e != cudaSuccess || cnt == 0)
        return fail(SS_ERR_DEVICE, 0, 0, 0, "no CUDA device available (%s); this library has no CPU fallback",
                    e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    if (g_devices.empty()) {
        const char* env = getenv("SNARK_SETUP_GPUS");
        if (env && *env) {
            std::string s(env);
            size_t pos = 0;
            while (pos < s.size()) {
                size_t c = s.find(',', pos);
                if (c == std::string::npos) c = s.size();
                g_devices.push_back(atoi(s.substr(pos, c - pos).c_str()));
                pos = c + 1;
            }
        } else {
            int cur = 0;
            cudaGetDevice(&cur);
            g_devices.push_back(cur);
        }
    }
    for (int d : g_devices)
        if (d < 0 || d >= cnt) return fail(SS_ERR_DEVICE, 0, 0, 0, "device %d out of range (count %d)", d, cnt);
    g_inited = true;
    return SS_OK;
}

// ---- lanes: stream + scratch, cached across calls -------------------------------------------------
struct Lane {
    int device = -1;
    cudaStream_t stream = nullptr;
    uint8_t* buf = nullptr;  // one slab, carved per use
    size_t cap = 0;
    bool busy = false;
    int prio = 0;  // 1: stream created with the device's highest priority (see lane_acquire)
};
std::vector<Lane*> g_lanes;

// ss_set_strict_unchecked_inputs: bases read without a subgroup check go through the reference's double-and-add
// instead of GLV / GLS (which presuppose the order-r subgroup), glv.cuh
std::atomic<int> g_strict_unchecked{0};
std::atomic<int> g_concurrent{-1};  // -1: take $SS_CONCURRENT_VECTORS (default on)
bool concurrent_vectors() {
    int v = g_concurrent.load();
    if (v < 0) {
        const char* e = getenv("SS_CONCURRENT_VECTORS");
        v = !(e && atoi(e) == 0);
        g_concurrent.store(v);
    }
    return v != 0;
}

// Elements per device tile.  k_scalar_mul does the same work in every thread, so its blocks finish in waves:
// the default is 16 whole waves of the G1 kernel (148 SMs x 4 resident blocks x 128 threads = 75 776
// elements per wave; the G2 kernel's waves are half that).  Measured (profiles/r01_ab_variants.md): wave quantisation is
// NOT visible (2^18: 251 ms, 4 waves: 248 ms), larger tiles win through fewer normalisation tails: 8 waves +1.3 % over 2^18
// (round 1), 16 waves another +0.85 % on the 2^22 contribute (1657.7 -> 1643.7 ms, profiles/r02_ab_variants.md).
// $SS_TILE_ELEMS / $SS_TILE_LOG2 override.
size_t tile_elems() {
    static size_t t = [] {
        if (const char* e = getenv("SS_TILE_ELEMS")) {
            long long v = atoll(e);
            if (v >= 256 && v <= (1ll << 24)) return (size_t)v;
        }
        if (const char* e = getenv("SS_TILE_LOG2")) {
            int l = atoi(e);
            if (l < 8) l = 8;
            if (l > 24) l = 24;
            return (size_t)1 << l;
        }
        return (size_t)16 * 75776;
    }();
    return t;
}

// prio = 1 asks for a lane whose stream has the device's highest scheduling priority: pending blocks of its kernels are
// dispatched before those of the normal lanes.  The verification loop gives it to the G2 vector, whose bucket reduction
// ends in a ~10 ms latency-bound tail (a handful of warps): finishing that vector FIRST hides the tail behind the
// throughput-bound kernels of the G1 vectors instead of leaving it exposed at the end of the call.
int lane_acquire(int device, size_t bytes, Lane** out, int prio = 0) {
    Lane* ln = nullptr;
    {
        std::lock_guard<std::mutex> lk(g_mu);
        // best fit: the smallest free slab that is large enough, else the largest free one (to grow);
        // keeps a 4 KB request from pinning a multi-GB slab and forcing other lanes to re-grow
        Lane* fit = nullptr;
        Lane* big = nullptr;
        for (Lane* l : g_lanes) {
            if (l->busy || l->device != device || l->prio != prio) continue;
            if (l->cap >= bytes && (!fit || l->cap < fit->cap)) fit = l;
            if (!big || l->cap > big->cap) big = l;
        }
        const size_t floor_b = std::max<size_t>(bytes, (size_t)1 << 20);
        if (fit && fit->cap <= 64 * floor_b) ln = fit;
        else if (!fit && big && bytes >= ((size_t)1 << 20)) ln = big;
        // otherwise (tiny request, only huge slabs free): open a new small lane
        if (!ln) {
            ln = new Lane();
            ln->device = device;
            ln->prio = prio;
            g_lanes.push_back(ln);
        }
        ln->busy = true;
    }
    // the caller's LaneGuard owns the lane from here on, so every error path below releases it
    *out = ln;
    CU(cudaSetDevice(device));
    if (!ln->stream) {
        int least = 0, greatest = 0;
        CU(cudaDeviceGetStreamPriorityRange(&least, &greatest));
        CU(cudaStreamCreateWithPriority(&ln->stream, cudaStreamNonBlocking, ln->prio ? greatest : least));
    }
    if (ln->cap < bytes) {
        if (ln->buf) CU(cudaFree(ln->buf));
        ln->buf = nullptr;
        ln->cap = 0;
        CU(cudaMalloc(&ln->buf, bytes));
        ln->cap = bytes;
    }
    return SS_OK;
}

void lane_release(Lane* l) {
    std::lock_guard<std::mutex> lk(g_mu);
    l->busy = false;
}

struct LaneGuard {
    Lane* l = nullptr;
    ~LaneGuard() {
        if (l) lane_release(l);
    }
};

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// carve helper
struct Carver {
    uint8_t* p;
    size_t off = 0;
    explicit Carver(uint8_t* base) : p(base) {}
    template <class T>
    T* take(size_t bytes) {
        T* r = reinterpret_cast<T*>(p + off);
        off += align_up(bytes, 256);
        return r;
    }
};

// scratch a tile of `t` elements needs (besides staged in/out bytes)
size_t scratch_bytes(const GroupOps& o, size_t t) {
    return align_up((size_t)3 * o.coord_words * 4 * t, 256) + align_up((size_t)o.coord_words * 4 * t, 256) +
           align_up((size_t)2 * o.coord_words * 4 * t, 256) + align_up(t, 256);
}

int decode_status(unsigned long long st, uint64_t base, const char* what) {
    if (st == STATUS_OK) return SS_OK;
    int code = (int)(st & 0xff);
    uint64_t idx = base + (st >> 8);
    return fail(code, idx, 0, 0, "%s: element %llu: error %d", what, (unsigned long long)idx, code);
}

uint32_t normalize_threads(uint64_t n) {
    // each thread batch-inverts up to 32 elements; at least one element per thread
    uint64_t t = (n + 31) / 32;
    if (t < 1024) t = std::min<uint64_t>(n, 1024);
    return (uint32_t)t;
}

// One vector of `n` elements.  host==true: in/out are host pointers and are staged tile by tile;
// host==false: in/out are device pointers of `device`.
struct VectorJob {
    const GroupOps* ops;
    const uint8_t* in;
    uint8_t* out;
    int in_c, out_c, check;
    uint64_t n;
    const uint8_t* exps;   // explicit scalars (host or device like in/out) or null
    const uint32_t* d_tab;
    uint64_t first_power;
    const uint32_t* d_coeff_m;
    int has_coeff;
    const char* what;
    bool exps_on_device = false;  // `exps` already lives in device memory even when in/out are host buffers
};

int run_vector_on(int device, const VectorJob& j, bool host, cudaStream_t user_stream) {
    if (j.n == 0) return SS_OK;
    const GroupOps& o = *j.ops;
    const size_t isz = j.in_c ? o.csize : o.usize, osz = j.out_c ? o.csize : o.usize;
    const size_t T = std::min<uint64_t>(tile_elems(), j.n);
    const size_t ntiles = (j.n + T - 1) / T;
    const int nl = (host && ntiles > 1) ? 2 : 1;
    size_t per_lane = scratch_bytes(o, T) + 256;
    const bool stage_exps = host && j.exps && !j.exps_on_device;
    const size_t fs = scalar_stride(o);
    std::vector<std::vector<uint8_t>> keep;
    if (host) per_lane += align_up(isz * T, 256) + align_up(osz * T, 256) + (stage_exps ? align_up(fs * T, 256) : 0);
    LaneGuard lg[2];
    for (int k = 0; k < nl; k++) {
        int rc = lane_acquire(device, per_lane + ntiles * 8 + 256, &lg[k].l);
        if (rc) return rc;
    }
    std::vector<unsigned long long> st(ntiles, STATUS_OK);
    // status words live at the head of lane 0's slab
    unsigned long long* d_status = reinterpret_cast<unsigned long long*>(lg[0].l->buf);
    cudaStream_t s0 = (!host && user_stream) ? user_stream : lg[0].l->stream;
    CU(cudaMemsetAsync(d_status, 0xff, ntiles * 8, s0));
    cudaEvent_t ev_init = nullptr;
    if (nl > 1) {
        CU(cudaEventCreateWithFlags(&ev_init, cudaEventDisableTiming));
        CU(cudaEventRecord(ev_init, s0));
        CU(cudaStreamWaitEvent(lg[1].l->stream, ev_init, 0));
    }
    const size_t status_bytes = align_up(ntiles * 8, 256);
    int rc = SS_OK;
    bool have_pending = false;
    uint8_t* pend_dst = nullptr;
    const uint8_t* pend_src = nullptr;
    size_t pend_bytes = 0;
    cudaStream_t pend_stream = nullptr;
    for (size_t t = 0; t < ntiles; t++) {
        const uint64_t e0 = t * T, cnt = std::min<uint64_t>(T, j.n - e0);
        Lane* ln = lg[t % nl].l;
        cudaStream_t s = (!host && user_stream) ? user_stream : ln->stream;
        Carver cv(ln->buf + ((t % nl) == 0 ? status_bytes : 0));
        uint32_t* jac = cv.take<uint32_t>((size_t)3 * o.coord_words * 4 * T);
        uint32_t* prefix = cv.take<uint32_t>((size_t)o.coord_words * 4 * T);
        uint32_t* aff = cv.take<uint32_t>((size_t)2 * o.coord_words * 4 * T);
        uint8_t* inf = cv.take<uint8_t>(T);
        const uint8_t* d_in;
        uint8_t* d_out;
        const uint8_t* d_exps = nullptr;
        if (host) {
            uint8_t* bi = cv.take<uint8_t>(isz * T);
            uint8_t* bo = cv.take<uint8_t>(osz * T);
            CU(cudaMemcpyAsync(bi, j.in + e0 * isz, cnt * isz, cudaMemcpyHostToDevice, s));
            if (stage_exps) {
                uint8_t* be = cv.take<uint8_t>(fs * T);
                const uint8_t* src = repack_scalars(o, j.exps + e0 * o.fr_bytes, cnt, keep);
                CU(cudaMemcpyAsync(be, src, cnt * fs, cudaMemcpyHostToDevice, s));
                d_exps = be;
            } else if (j.exps) {
                d_exps = j.exps + e0 * fs;  // already on the device, word stride
            }
            d_in = bi;
            d_out = bo;
        } else {
            d_in = j.in + e0 * isz;
            d_out = j.out + e0 * osz;
            if (j.exps) d_exps = j.exps + e0 * fs;
        }
        DecodeArgs da;
        da.in = reinterpret_cast<const uint32_t*>(d_in);
        da.in_compressed = j.in_c;
        da.check = j.check;
        da.n = cnt;
        da.aff = aff;
        da.inf = inf;
        da.status = d_status + t;
        { ProfScope ps("k_decode", o.name, cnt, s); o.decode(da, s); }
        ScalarMulArgs a;
        a.aff = aff;
        a.inf = inf;
        a.n = cnt;
        a.exps = reinterpret_cast<const uint32_t*>(d_exps);
        a.tau_tab = j.d_tab;
        a.first_power = j.first_power + e0;
        a.coeff_m = j.d_coeff_m;
        a.has_coeff = j.has_coeff;
        a.jac = jac;
        a.plain_ladder = (g_strict_unchecked.load() && (j.check == SS_CHECK_NO || j.check == SS_CHECK_ONLY_NON_ZERO)) ? 1 : 0;
        { ProfScope ps("k_scalar_mul", o.name, cnt, s); o.scalar_mul(a, s); }
        NormalizeArgs na;
        na.jac = jac;
        na.n = cnt;
        na.prefix = prefix;
        na.out = reinterpret_cast<uint32_t*>(d_out);
        na.out_compressed = j.out_c;
        na.threads = normalize_threads(cnt);
        { ProfScope ps("k_normalize_encode", o.name, cnt, s); o.normalize_encode(na, s); }
        // Output copies run ONE TILE BEHIND: a device-to-host copy into PAGEABLE memory (the callers' mmaps) blocks the
        // issuing thread until the tile's kernels have finished, so issuing it right here would keep tile t + 1 (other
        // lane) from being enqueued until tile t is completely done.  Its slab region is safe: the lane is reused by
        // tile t + 2, enqueued after the copy on the same stream.  For pinned buffers the order is immaterial.
        if (host) {
            if (have_pending) CU(cudaMemcpyAsync(pend_dst, pend_src, pend_bytes, cudaMemcpyDeviceToHost, pend_stream));
            pend_dst = j.out + e0 * osz;
            pend_src = d_out;
            pend_bytes = cnt * osz;
            pend_stream = s;
            have_pending = true;
        }
    }
    if (have_pending) CU(cudaMemcpyAsync(pend_dst, pend_src, pend_bytes, cudaMemcpyDeviceToHost, pend_stream));
    CU(cudaGetLastError());
    for (int k = 0; k < nl; k++) CU(cudaStreamSynchronize((!host && user_stream) ? user_stream : lg[k].l->stream));
    if (ev_init) cudaEventDestroy(ev_init);
    CU(cudaMemcpy(st.data(), d_status, ntiles * 8, cudaMemcpyDeviceToHost));
    prof_flush();
    for (size_t t = 0; t < ntiles && rc == SS_OK; t++) rc = decode_status(st[t], t * T, j.what);
    return rc;
}

// scalar context: uploads tau / coefficients and builds the tau^(2^j) table on the device
struct ScalarSetup {
    uint8_t* slab = nullptr;
    uint32_t* d_tab = nullptr;
    uint32_t* d_coeff_m[3] = {nullptr, nullptr, nullptr};
    ~ScalarSetup() {
        if (slab) cudaFree(slab);
    }
    // coeffs[k] may be null -> Montgomery one
    int init(const GroupOps& o, const uint8_t* tau, const uint8_t* const coeffs[3], cudaStream_t s) {
        const size_t fb = o.fr_bytes, fw = o.fr_words;
        const size_t tab_b = align_up(64 * fw * 4, 256), el_b = align_up(fw * 4, 256);
        CU(cudaMalloc(&slab, tab_b + 3 * el_b + 4 * el_b));
        CU(cudaMemsetAsync(slab, 0, tab_b + 3 * el_b + 4 * el_b, s));  // scalars of 95 bytes leave a partial top word
        d_tab = reinterpret_cast<uint32_t*>(slab);
        uint8_t* p = slab + tab_b;
        for (int k = 0; k < 3; k++) d_coeff_m[k] = reinterpret_cast<uint32_t*>(p + k * el_b);
        uint8_t* raw = p + 3 * el_b;  // tau, c0, c1, c2 canonical
        std::vector<uint8_t> zero(fb, 0);
        CU(cudaMemcpyAsync(raw, tau ? tau : zero.data(), fb, cudaMemcpyHostToDevice, s));
        for (int k = 0; k < 3; k++)
            if (coeffs[k]) CU(cudaMemcpyAsync(raw + (k + 1) * el_b, coeffs[k], fb, cudaMemcpyHostToDevice, s));
        CU(cudaStreamSynchronize(s));  // `zero` goes out of scope
        for (int k = 0; k < 3; k++)
            o.prepare_scalars(reinterpret_cast<uint32_t*>(raw),
                              coeffs[k] ? reinterpret_cast<uint32_t*>(raw + (k + 1) * el_b) : nullptr,
                              d_tab, d_coeff_m[k], s);
        CU(cudaGetLastError());
        CU(cudaStreamSynchronize(s));
        return SS_OK;
    }
};

// the scalar-field modulus r of a curve, little-endian u32 limbs
const uint32_t* scalar_modulus(int curve, int* n) {
    static const uint32_t r_bls[8] = {0x00000001u, 0x0a118000u, 0xd0000001u, 0x59aa76feu, 0x5c37b001u, 0x60b44d1eu, 0x9a2ca556u, 0x12ab655eu};
    static const uint32_t r_bw6[12] = {0x00000001u, 0x8508c000u, 0x30000000u, 0x170b5d44u, 0xba094800u, 0x1ef3622fu, 0x00f5138fu, 0x1a22d9f3u, 0x6ca1493bu, 0xc63b05c0u, 0x17c510eau, 0x01ae3a46u};
    static uint32_t r_mnt[2][24];
    static const bool init = [] {  // MNT4 Fr = Mnt753R, MNT6 Fr = Mnt753Q (constants_gen.cuh)
        for (int i = 0; i < 24; i++) {
            r_mnt[0][i] = Mnt753R::mod(i);
            r_mnt[1][i] = Mnt753Q::mod(i);
        }
        return true;
    }();
    (void)init;
    switch (curve) {
        case SS_CURVE_BLS12_377: *n = 8; return r_bls;
        case SS_CURVE_BW6_761: *n = 12; return r_bw6;
        case SS_CURVE_MNT4_753: *n = 24; return r_mnt[0];
        case SS_CURVE_MNT6_753: *n = 24; return r_mnt[1];
    }
    *n = 0;
    return nullptr;
}

bool scalar_is_canonical(int curve, const uint8_t* s) {
    int n;
    const uint32_t* r = scalar_modulus(curve, &n);
    if (!r) return false;
    const GroupOps* o = group_ops(curve, SS_G1);
    uint32_t w[24] = {0};
    memcpy(w, s, o->fr_bytes);  // 95-byte scalars: the top word is zero-extended
    for (int i = n - 1; i >= 0; i--) {
        if (w[i] < r[i]) return true;
        if (w[i] > r[i]) return false;
    }
    return false;
}

// [start, end) of part `part` of `parts` equal contiguous parts of n elements (the first n % parts parts get one more)
void part_range(uint64_t n, uint64_t part, uint64_t parts, uint64_t* s0, uint64_t* e0) {
    const uint64_t base = n / parts, rem = n % parts;
    *s0 = part * base + std::min<uint64_t>(part, rem);
    *e0 = *s0 + base + (part < rem ? 1 : 0);
}

// Runs job(0) .. job(n - 1) and returns the first failure.  When n == 1 or !parallel the jobs run in order on the
// calling thread and stop at the first failure; otherwise each gets a thread of its own.  g_err is thread-local, so a
// failing thread's record is copied out, and after the join the lowest-indexed failure is restored and returned.
template <class F>
int run_jobs(int n, bool parallel, F job) {
    if (n == 1 || !parallel) {
        for (int i = 0; i < n; i++)
            if (int rc = job(i)) return rc;
        return SS_OK;
    }
    std::vector<int> rcs(n, SS_OK);
    std::vector<ss_error_info> errs(n);
    std::vector<std::thread> th;
    for (int i = 0; i < n; i++)
        th.emplace_back([&, i] {
            if ((rcs[i] = job(i))) errs[i] = g_err;
        });
    for (auto& t : th) t.join();
    for (int i = 0; i < n; i++)
        if (rcs[i]) {
            g_err = errs[i];
            return rcs[i];
        }
    return SS_OK;
}

// The five vectors of a phase-1 buffer, in buffer order, with their groups
const int kVecGroup[5] = {SS_G1, SS_G2, SS_G1, SS_G1, SS_G2};
const char* const kVecName[5] = {"tau_g1", "tau_g2", "alpha_g1", "beta_g1", "beta_g2"};

// The phase-1 buffer of one chunk, split / split_mut (buffers.rs:246-341): the 64-byte hash, then
// [tau_g1][tau_g2][alpha_g1][beta_g1][beta_g2].  Marlin has tau_g1 and, in the buffer of chunk 0 only, k+2 tau_g2 and
// 3+3k alpha_g1 elements; its beta counts are zero.  Phase1Parameters::new / chunk_sizes (parameters.rs:115-294) give
// the counts.
struct Phase1Layout {
    uint64_t powers_length, powers_g1_length, g1_chunk_size, other_chunk_size;
    struct Vector {
        const GroupOps* ops;
        int group;
        uint64_t size, count, off;  // bytes per element, elements, byte offset in the buffer
        const char* name;
    } v[5];
    uint64_t end;  // bytes of the buffer, without the public key
};

int phase1_layout(const ss_phase1_params* p, int compressed, Phase1Layout* L) {
    if (!p) return fail(SS_ERR_INVALID_ARGUMENT, 0, 0, 0, "null argument");
    const GroupOps* g1 = group_ops(p->curve, SS_G1);
    const GroupOps* g2 = group_ops(p->curve, SS_G2);
    if (!g1 || !g2) return fail(SS_ERR_INVALID_ARGUMENT, 0, 0, 0, "unknown curve %d", p->curve);
    if (p->total_size_in_log2 == 0 || p->total_size_in_log2 > 40)
        return fail(SS_ERR_INVALID_ARGUMENT, 0, 0, 0, "bad power %u", p->total_size_in_log2);
    const bool groth16 = p->proving_system == SS_GROTH16;
    const uint64_t k = p->total_size_in_log2, pl = 1ull << k, pg1 = (pl << 1) - 1;
    const uint64_t upper = groth16 ? pg1 : pl;
    uint64_t start = 0, end = upper;
    if (p->contribution_mode == SS_MODE_CHUNKED) {
        start = p->chunk_index * p->chunk_size;
        end = (p->chunk_index + 1) * p->chunk_size;
        if (p->chunk_size == 0 || start >= upper) return fail(SS_ERR_INVALID_CHUNK, 0, 0, 0, "chunk out of range");
    }
    L->powers_length = pl;
    L->powers_g1_length = pg1;
    L->g1_chunk_size = std::min(end, upper) - start;
    L->other_chunk_size = groth16 && start < pl ? std::min(end, pl) - start : 0;
    // Marlin's short tau_g2 / alpha_g1 vectors live in the buffer of chunk_index 0 — the ONE predicate the reference
    // uses for the sizes (parameters.rs:152-160), the buffer split (buffers.rs:151,220,274,324) and the computation
    // (computation.rs:198); full-mode callers pass chunk_index = 0.
    const bool chunk0 = p->chunk_index == 0;
    const uint64_t n2 = L->other_chunk_size;
    const uint64_t cnt[5] = {L->g1_chunk_size, groth16 ? n2 : (chunk0 ? k + 2 : 0), groth16 ? n2 : (chunk0 ? 3 + 3 * k : 0),
                             groth16 ? n2 : 0, groth16 ? 1u : 0u};
    uint64_t off = 64;
    for (int v = 0; v < 5; v++) {
        Phase1Layout::Vector& e = L->v[v];
        e.group = kVecGroup[v];
        e.ops = e.group == SS_G1 ? g1 : g2;
        e.size = compressed ? e.ops->csize : e.ops->usize;
        e.count = cnt[v];
        e.off = off;
        e.name = kVecName[v];
        off += e.count * e.size;
    }
    L->end = off;
    return SS_OK;
}

// SS_ERR_INVALID_LENGTH unless `len` bytes hold the buffer of layout `L`
int check_length(const Phase1Layout& L, uint64_t len, const char* what) {
    return len < L.end ? fail(SS_ERR_INVALID_LENGTH, 0, L.end, len, "%s", what) : SS_OK;
}

// The (s, sx) pairs blob of the four ratio-checked vectors: slot v holds s || sx of vector v, uncompressed, so
// 4 x (s || sx) in the order G1, G2, G1, G1.  pair_slot(curve, 4) is the size of the blob, 0 for an unknown curve.
size_t pair_slot(int curve, int v) {
    size_t off = 0;
    for (int u = 0; u < v; u++) {
        const GroupOps* o = group_ops(curve, kVecGroup[u]);
        if (!o) return 0;
        off += 2 * (size_t)o->usize;
    }
    return off;
}

int phase1_sizes(const ss_phase1_params* p, ss_phase1_sizes* o) {
    if (!p || !o) return fail(SS_ERR_INVALID_ARGUMENT, 0, 0, 0, "null argument");
    Phase1Layout u, c;
    int rc;
    if ((rc = phase1_layout(p, 0, &u)) || (rc = phase1_layout(p, 1, &c))) return rc;
    o->powers_length = u.powers_length;
    o->powers_g1_length = u.powers_g1_length;
    o->g1_chunk_size = u.g1_chunk_size;
    o->other_chunk_size = u.other_chunk_size;
    o->hash_size = 64;
    o->public_key_size = 3 * (uint64_t)u.v[1].ops->csize + 6 * (uint64_t)u.v[0].ops->csize;
    o->accumulator_size = u.end;
    o->contribution_size = c.end + o->public_key_size;
    return SS_OK;
}

// Phase1::computation (phase1/src/computation.rs:40-302), Groth16 and Marlin
int phase1_computation_impl(const ss_phase1_params* p, const uint8_t* input, size_t input_len, uint8_t* output,
                            size_t output_len, int cin, int cout, int check, const uint8_t* tau,
                            const uint8_t* alpha, const uint8_t* beta, bool host, cudaStream_t user_stream,
                            uint32_t shard_index = 0, uint32_t shard_count = 1) {
    if (!p || !input || !output || !tau || !alpha || (!beta && p->proving_system != SS_MARLIN))
        return fail(SS_ERR_INVALID_ARGUMENT, 0, 0, 0, "null argument");
    if (shard_count == 0 || shard_index >= shard_count)
        return fail(SS_ERR_INVALID_ARGUMENT, 0, 0, 0, "shard %u of %u", shard_index, shard_count);
    if (check < 0 || check > 3) return fail(SS_ERR_INVALID_ARGUMENT, 0, 0, 0, "bad check mode %d", check);
    Phase1Layout li, lo;  // input, output
    int rc;
    if ((rc = phase1_layout(p, cin, &li)) || (rc = phase1_layout(p, cout, &lo))) return rc;
    if ((rc = check_length(li, input_len, "input buffer too short"))) return rc;
    if ((rc = check_length(lo, output_len, "output buffer too short"))) return rc;
    const bool marlin = p->proving_system == SS_MARLIN;
    if (marlin) beta = nullptr;  // Marlin has no beta
    for (const uint8_t* s : {tau, alpha, beta})
        if (s && !scalar_is_canonical(p->curve, s)) return fail(SS_ERR_INVALID_DATA, 0, 0, 0, "scalar >= r");
    if ((rc = ensure_init())) return rc;
    const GroupOps& g1 = *li.v[0].ops;
    const uint64_t first = p->contribution_mode == SS_MODE_CHUNKED ? p->chunk_index * p->chunk_size : 0;
    const bool concurrent = concurrent_vectors();

    // One worker per device.  Every vector is cut into shard_count * D equal contiguous parts (SURVEY.md §8e:
    // balance by work, not by index — indices >= 2^k only carry one G1 element); this call owns parts
    // [shard_index * D, (shard_index + 1) * D), one per device.  Element i of a part still gets tau^(first + i)
    // because each part passes its own first power.  No inter-device / inter-process traffic.
    const int D = host ? (int)g_devices.size() : 1;
    const uint64_t parts = (uint64_t)shard_count * D;
    return run_jobs(D, true, [&](int di) -> int {
        const int device = host ? g_devices[di] : g_devices[0];
        CU(cudaSetDevice(device));
        // beta_g2 <- beta * beta_g2 (computation.rs:42-50) and Marlin's tau_g2 / alpha_g1 are not split: the owner of
        // part 0 does them whole.  The scalars of Marlin's two (computation.rs:195-302: inverse degree-bound powers
        // etc.) are produced by k_marlin_scalars and applied through the explicit-exponent path.
        const bool part0 = di == 0 && shard_index == 0;
        const uint64_t n_g2 = part0 && marlin ? li.v[1].count : 0, n_al = part0 && marlin ? li.v[2].count : 0;
        LaneGuard setup_lane;
        int r = lane_acquire(device, 4096 + (n_g2 + n_al) * scalar_stride(g1), &setup_lane.l);
        if (r) return r;
        ScalarSetup sc;
        const uint8_t* coeffs[3] = {nullptr, alpha, beta};
        if ((r = sc.init(g1, tau, coeffs, setup_lane.l->stream))) return r;
        uint8_t *d_g2s = nullptr, *d_als = nullptr;
        if (n_g2 + n_al) {
            d_g2s = setup_lane.l->buf;
            d_als = d_g2s + align_up(n_g2 * scalar_stride(g1), 256);
            g1.marlin_scalars(sc.d_tab, li.powers_length, (int)p->total_size_in_log2, reinterpret_cast<uint32_t*>(d_g2s),
                              reinterpret_cast<uint32_t*>(d_als), setup_lane.l->stream);
            CU(cudaGetLastError());
            CU(cudaStreamSynchronize(setup_lane.l->stream));
        }
        const uint8_t* exps[5] = {nullptr, d_g2s, d_als, nullptr, nullptr};
        const uint32_t* cm[5] = {sc.d_coeff_m[0], sc.d_coeff_m[0], sc.d_coeff_m[1], sc.d_coeff_m[2], sc.d_coeff_m[2]};
        const int hc[5] = {0, 0, 1, 1, 1};
        // The five vectors run CONCURRENTLY, one host thread + lane (stream, scratch) each: the
        // low-occupancy tails (batch normalisation, the single beta_g2 element) of one vector overlap the
        // scalar multiplications of another.  SS_CONCURRENT_VECTORS=0 restores the sequential order.
        auto one_vector = [&](int v) -> int {
            cudaSetDevice(device);
            const Phase1Layout::Vector &vi = li.v[v], &vo = lo.v[v];
            const bool split = v == 0 || (!marlin && v < 4);  // powers of tau: split into parts
            uint64_t s0 = 0, e0 = vi.count;
            if (split) part_range(vi.count, (uint64_t)shard_index * D + di, parts, &s0, &e0);
            else if (!part0) return SS_OK;
            VectorJob job = {vi.ops, input + vi.off + s0 * vi.size, output + vo.off + s0 * vo.size, cin, cout, check,
                             e0 - s0, exps[v], sc.d_tab, split ? first + s0 : 0, cm[v], hc[v], vi.name, true};
            int rv = run_vector_on(device, job, host, concurrent ? nullptr : user_stream);
            if (rv) g_err.index += s0;  // report vector-relative indices
            return rv;
        };
        if (concurrent && user_stream) CU(cudaStreamSynchronize(user_stream));  // work enqueued before the call comes first
        return run_jobs(5, concurrent, one_vector);
    });
}

}  // namespace

// =====================================================================================================
#include "api_ratio.inl"

extern "C" {

const char* ss_version(void) { return "snark-setup-b200 0.1 (sm_100a)"; }

void ss_last_error(ss_error_info* out) {
    if (out) *out = g_err;
}

int ss_init(const int* devices, int n_devices) {
    {
        std::lock_guard<std::mutex> lk(g_mu);
        g_devices.clear();
        for (int i = 0; i < n_devices; i++) g_devices.push_back(devices[i]);
        g_inited = false;
    }
    return ensure_init();
}

void ss_shutdown(void) {
    std::lock_guard<std::mutex> lk(g_mu);
    for (Lane* l : g_lanes) {
        cudaSetDevice(l->device);
        if (l->buf) cudaFree(l->buf);
        if (l->stream) cudaStreamDestroy(l->stream);
        delete l;
    }
    g_lanes.clear();
    g_inited = false;
}

void ss_profile_enable(int on) {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    g_prof_on = on != 0;
}

void ss_profile_reset(void) {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    g_prof.clear();
    g_launches.store(0);
}

uint64_t ss_profile_launches(void) { return g_launches.load(); }

int ss_profile_read(ss_profile_entry* out, int max_entries) {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    int n = 0;
    for (auto& a : g_prof) {
        if (n >= max_entries) break;
        memset(&out[n], 0, sizeof(out[n]));
        snprintf(out[n].name, sizeof(out[n].name), "%s", a.name.c_str());
        out[n].launches = a.launches;
        out[n].elements = a.elements;
        out[n].ms = a.ms;
        n++;
    }
    return n;
}

void ss_set_concurrent_vectors(int on) { g_concurrent.store(on ? 1 : 0); }

void ss_set_strict_unchecked_inputs(int on) { g_strict_unchecked.store(on ? 1 : 0); }

int ss_device_count(void) {
    int c = 0;
    if (cudaGetDeviceCount(&c) != cudaSuccess) return 0;
    return c;
}

size_t ss_element_size(int curve, int group, int compressed) {
    const GroupOps* o = group_ops(curve, group);
    if (!o) return 0;
    return compressed ? o->csize : o->usize;
}

size_t ss_scalar_size(int curve) {
    const GroupOps* o = group_ops(curve, SS_G1);
    return o ? o->fr_bytes : 0;
}

int ss_generate_powers_of_tau(int curve, const uint8_t* tau, uint64_t start, uint64_t end, uint8_t* out) {
    const GroupOps* o = group_ops(curve, SS_G1);
    if (!o || !tau || (!out && end > start)) return fail(SS_ERR_INVALID_ARGUMENT, 0, 0, 0, "bad argument");
    if (end <= start) return SS_OK;
    if (!scalar_is_canonical(curve, tau)) return fail(SS_ERR_INVALID_DATA, 0, 0, 0, "tau >= r");
    int rc = ensure_init();
    if (rc) return rc;
    const int device = g_devices[0];
    const uint64_t n = end - start;
    LaneGuard lg;
    const size_t fs = scalar_stride(*o), fb = o->fr_bytes;
    if ((rc = lane_acquire(device, n * fs + 256, &lg.l))) return rc;
    ScalarSetup sc;
    const uint8_t* coeffs[3] = {nullptr, nullptr, nullptr};
    if ((rc = sc.init(*o, tau, coeffs, lg.l->stream))) return rc;
    o->powers(sc.d_tab, start, n, reinterpret_cast<uint32_t*>(lg.l->buf), lg.l->stream);
    CU(cudaGetLastError());
    if (fs == fb) {
        CU(cudaMemcpyAsync(out, lg.l->buf, n * fb, cudaMemcpyDeviceToHost, lg.l->stream));
        CU(cudaStreamSynchronize(lg.l->stream));
    } else {  // device words -> packed ceil(bits / 8)-byte scalars
        std::vector<uint8_t> tmp(n * fs);
        CU(cudaMemcpyAsync(tmp.data(), lg.l->buf, n * fs, cudaMemcpyDeviceToHost, lg.l->stream));
        CU(cudaStreamSynchronize(lg.l->stream));
        for (uint64_t i = 0; i < n; i++) memcpy(out + i * fb, tmp.data() + i * fs, fb);
    }
    return SS_OK;
}

int ss_apply_powers(int curve, int group, const uint8_t* in, int in_compressed, int in_check, uint8_t* out,
                    int out_compressed, size_t n, const uint8_t* powers, const uint8_t* tau, uint64_t first_power,
                    const uint8_t* coeff) {
    const GroupOps* o = group_ops(curve, group);
    if (!o) return fail(SS_ERR_INVALID_ARGUMENT, 0, 0, 0, "unknown curve/group %d/%d", curve, group);
    if (n == 0) return SS_OK;
    if (!in || !out || (!powers && !tau)) return fail(SS_ERR_INVALID_ARGUMENT, 0, 0, 0, "null argument");
    if (in_check < 0 || in_check > 3) return fail(SS_ERR_INVALID_ARGUMENT, 0, 0, 0, "bad check mode");
    if (tau && !powers && !scalar_is_canonical(curve, tau)) return fail(SS_ERR_INVALID_DATA, 0, 0, 0, "tau >= r");
    if (coeff && !scalar_is_canonical(curve, coeff)) return fail(SS_ERR_INVALID_DATA, 0, 0, 0, "coeff >= r");
    if (powers)
        for (size_t i = 0; i < n; i++)
            if (!scalar_is_canonical(curve, powers + i * o->fr_bytes))
                return fail(SS_ERR_INVALID_DATA, i, 0, 0, "scalar %zu >= r", i);
    int rc = ensure_init();
    if (rc) return rc;
    const int device = g_devices[0];
    LaneGuard lg;
    if ((rc = lane_acquire(device, 4096, &lg.l))) return rc;
    ScalarSetup sc;
    const uint8_t* coeffs[3] = {coeff, nullptr, nullptr};
    if ((rc = sc.init(*o, powers ? nullptr : tau, coeffs, lg.l->stream))) return rc;
    VectorJob j = {o, in, out, in_compressed, out_compressed, in_check, n, powers, sc.d_tab, first_power,
                   sc.d_coeff_m[0], coeff ? 1 : 0, "apply_powers"};
    return run_vector_on(device, j, true, nullptr);
}

int ss_batch_exp(int curve, int group, uint8_t* bases, size_t n, const uint8_t* exps, size_t n_exps,
                 const uint8_t* coeff) {
    if (n != n_exps) return fail(SS_ERR_INVALID_LENGTH, 0, n, n_exps, "bases.len() != exps.len()");
    return ss_apply_powers(curve, group, bases, 0, SS_CHECK_NO, bases, 0, n, exps, nullptr, 0, coeff);
}

int ss_batch_mul(int curve, int group, uint8_t* bases, size_t n, const uint8_t* coeff) {
    if (!coeff) return fail(SS_ERR_INVALID_ARGUMENT, 0, 0, 0, "null coeff");
    // every exponent equal to coeff == tau^0 * coeff
    const GroupOps* o = group_ops(curve, group);
    if (!o) return fail(SS_ERR_INVALID_ARGUMENT, 0, 0, 0, "unknown curve/group");
    std::vector<uint8_t> one(o->fr_bytes, 0);
    one[0] = 1;
    if (n == 0) return SS_OK;
    if (!bases) return fail(SS_ERR_INVALID_ARGUMENT, 0, 0, 0, "null bases");
    if (!scalar_is_canonical(curve, coeff)) return fail(SS_ERR_INVALID_DATA, 0, 0, 0, "coeff >= r");
    int rc = ensure_init();
    if (rc) return rc;
    const int device = g_devices[0];
    LaneGuard lg;
    if ((rc = lane_acquire(device, 4096, &lg.l))) return rc;
    ScalarSetup sc;
    const uint8_t* coeffs[3] = {coeff, nullptr, nullptr};
    if ((rc = sc.init(*o, one.data(), coeffs, lg.l->stream))) return rc;
    // first_power = 0 for every element: use a zero-stride trick by exponent 0 -> tau^0; the kernel
    // adds the element index, so pass tau = 1 (1^i = 1).
    VectorJob j = {o, bases, bases, 0, 0, SS_CHECK_NO, n, nullptr, sc.d_tab, 0, sc.d_coeff_m[0], 1, "batch_mul"};
    return run_vector_on(device, j, true, nullptr);
}

// decode (+ optional subgroup r-mul) (+ optional re-encode) over host buffers, tile by tile
static int transcode_impl(int curve, int group, const uint8_t* in, int in_compressed, int check, uint8_t* out,
                          int out_compressed, size_t n, bool rmul_subgroup) {
    const GroupOps* o = group_ops(curve, group);
    if (!o) return fail(SS_ERR_INVALID_ARGUMENT, 0, 0, 0, "unknown curve/group");
    if (n == 0) return SS_OK;
    if (!in) return fail(SS_ERR_INVALID_ARGUMENT, 0, 0, 0, "null input");
    if (check < 0 || check > 3) return fail(SS_ERR_INVALID_ARGUMENT, 0, 0, 0, "bad check mode");
    int rc = ensure_init();
    if (rc) return rc;
    const int device = g_devices[0];
    const size_t isz = in_compressed ? o->csize : o->usize, osz = out_compressed ? o->csize : o->usize;
    const size_t T = std::min<size_t>(tile_elems(), n);
    LaneGuard lg;
    const size_t aff_b = align_up((size_t)2 * o->coord_words * 4 * T, 256);
    if ((rc = lane_acquire(device, 256 + align_up(isz * T, 256) + align_up(osz * T, 256) + aff_b + align_up(T, 256), &lg.l)))
        return rc;
    cudaStream_t s = lg.l->stream;
    Carver cv(lg.l->buf);
    unsigned long long* d_status = cv.take<unsigned long long>(16);
    uint8_t* bi = cv.take<uint8_t>(isz * T);
    uint8_t* bo = cv.take<uint8_t>(osz * T);
    uint32_t* aff = cv.take<uint32_t>((size_t)2 * o->coord_words * 4 * T);
    uint8_t* inf = cv.take<uint8_t>(T);
    for (size_t e0 = 0; e0 < n; e0 += T) {
        const size_t cnt = std::min(T, n - e0);
        CU(cudaMemsetAsync(d_status, 0xff, 16, s));
        CU(cudaMemcpyAsync(bi, in + e0 * isz, cnt * isz, cudaMemcpyHostToDevice, s));
        DecodeArgs da = {reinterpret_cast<const uint32_t*>(bi), in_compressed, check, cnt, aff, inf, d_status};
        { ProfScope ps("k_decode", o->name, cnt, s); o->decode(da, s); }
        if (rmul_subgroup) {
            SubgroupArgs sa = {aff, inf, cnt, d_status + 1, cnt, in_compressed ? 0 : 1};
            ProfScope ps("k_subgroup", o->name, cnt, s);
            o->subgroup(sa, s);
        }
        if (out) {
            EncodeArgs ea = {aff, inf, cnt, reinterpret_cast<uint32_t*>(bo), out_compressed, cnt};
            ProfScope ps("k_encode", o->name, cnt, s);
            o->encode(ea, s);
        }
        CU(cudaGetLastError());
        unsigned long long st[2];
        CU(cudaMemcpyAsync(st, d_status, 16, cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
        prof_flush();
        if ((rc = decode_status(st[0], e0, "read_batch"))) return rc;
        if ((rc = decode_status(st[1], e0, "check_subgroup"))) return rc;
        if (out) {
            CU(cudaMemcpyAsync(out + e0 * osz, bo, cnt * osz, cudaMemcpyDeviceToHost, s));
            CU(cudaStreamSynchronize(s));
        }
    }
    return SS_OK;
}

int ss_transcode(int curve, int group, const uint8_t* in, int in_compressed, int check, uint8_t* out,
                 int out_compressed, size_t n) {
    return transcode_impl(curve, group, in, in_compressed, check, out, out_compressed, n, false);
}

int ss_check_subgroup(int curve, int group, const uint8_t* in, int compressed, size_t n, int subgroup_mode) {
    if (subgroup_mode < 0 || subgroup_mode > 3) return fail(SS_ERR_INVALID_ARGUMENT, 0, 0, 0, "bad subgroup mode");
    // elements were read by the caller with Validate::No; every mode but `No` collapses to the direct
    // r-multiplication (setup-utils/src/elements.rs:129-144)
    return transcode_impl(curve, group, in, compressed, SS_CHECK_NO, nullptr, 0, n, subgroup_mode != SS_SUBGROUP_NO);
}

// ---- accumulator re-layout: aggregation / split / decompress ----------------------------------------
// All three are read_batch(CheckForCorrectness) -> write_batch streams over the five vectors with different
// source / destination offsets (phase1/src/aggregation.rs:11-180,189-353; helpers/accumulator.rs:182-301).
static int copy_vectors(int curve, const uint8_t* src, const uint64_t* so, int src_c, uint8_t* dst, const uint64_t* dof,
                        int dst_c, const uint64_t* cnt, int check) {
    for (int v = 0; v < 5; v++) {
        if (!cnt[v]) continue;
        int rc = transcode_impl(curve, kVecGroup[v], src + so[v], src_c, check, dst + dof[v], dst_c, cnt[v], false);
        if (rc) return rc;
    }
    return SS_OK;
}

static int chunk_vs_full(const ss_phase1_params* cp, int compressed_chunk, int compressed_full, size_t chunk_len, size_t full_len,
                         uint64_t* coff, uint64_t* foff, uint64_t* cnt) {
    if (!cp) return fail(SS_ERR_INVALID_ARGUMENT, 0, 0, 0, "null argument");
    if (cp->proving_system != SS_GROTH16) return fail(SS_ERR_INVALID_ARGUMENT, 0, 0, 0, "only the Groth16 layout is implemented");
    if (cp->contribution_mode != SS_MODE_CHUNKED) return fail(SS_ERR_INVALID_ARGUMENT, 0, 0, 0, "chunk parameters expected");
    ss_phase1_params fp = *cp;
    fp.contribution_mode = SS_MODE_FULL;
    fp.chunk_index = 0;
    Phase1Layout c, f;
    int rc;
    if ((rc = phase1_layout(cp, compressed_chunk, &c)) || (rc = phase1_layout(&fp, compressed_full, &f))) return rc;
    if ((rc = check_length(c, chunk_len, "chunk buffer too short"))) return rc;
    if ((rc = check_length(f, full_len, "full buffer too short"))) return rc;
    // split_at_chunk(_mut): the chunk starts chunk_index * chunk_size elements into every vector
    const uint64_t first = cp->chunk_index * cp->chunk_size;
    for (int v = 0; v < 5; v++) {
        coff[v] = c.v[v].off;
        foff[v] = f.v[v].off + (v < 4 ? first * f.v[v].size : 0);
        cnt[v] = c.v[v].count;
    }
    cnt[4] = cp->chunk_index == 0 ? 1 : 0;  // beta_g2 travels with chunk 0 (aggregation.rs:103-111)
    return SS_OK;
}

int ss_phase1_aggregate_chunk(const ss_phase1_params* chunk_params, const uint8_t* chunk, size_t chunk_len, int compressed_chunk,
                              uint8_t* full, size_t full_len, int compressed_full) {
    uint64_t coff[5], foff[5], cnt[5];
    int rc = chunk_vs_full(chunk_params, compressed_chunk, compressed_full, chunk_len, full_len, coff, foff, cnt);
    if (rc) return rc;
    if (!chunk || !full) return fail(SS_ERR_INVALID_ARGUMENT, 0, 0, 0, "null buffer");
    return copy_vectors(chunk_params->curve, chunk, coff, compressed_chunk, full, foff, compressed_full, cnt, SS_CHECK_NO);
}

int ss_phase1_split_chunk(const ss_phase1_params* chunk_params, const uint8_t* full, size_t full_len, int compressed_full,
                          uint8_t* chunk, size_t chunk_len, int compressed_chunk) {
    uint64_t coff[5], foff[5], cnt[5];
    int rc = chunk_vs_full(chunk_params, compressed_chunk, compressed_full, chunk_len, full_len, coff, foff, cnt);
    if (rc) return rc;
    if (!chunk || !full) return fail(SS_ERR_INVALID_ARGUMENT, 0, 0, 0, "null buffer");
    cnt[4] = 1;  // every chunk file gets beta_g2 (aggregation.rs:278-284 writes it unconditionally)
    return copy_vectors(chunk_params->curve, full, foff, compressed_full, chunk, coff, compressed_chunk, cnt, SS_CHECK_NO);
}

int ss_phase1_decompress(const ss_phase1_params* p, const uint8_t* in, size_t in_len, int check, uint8_t* out, size_t out_len) {
    if (!p || !in || !out) return fail(SS_ERR_INVALID_ARGUMENT, 0, 0, 0, "null argument");
    if (p->proving_system != SS_GROTH16) return fail(SS_ERR_INVALID_ARGUMENT, 0, 0, 0, "only the Groth16 layout is implemented");
    if (check < 0 || check > 3) return fail(SS_ERR_INVALID_ARGUMENT, 0, 0, 0, "bad check mode");
    Phase1Layout c, u;
    int rc;
    if ((rc = phase1_layout(p, 1, &c)) || (rc = phase1_layout(p, 0, &u))) return rc;
    if ((rc = check_length(c, in_len, "compressed buffer too short"))) return rc;
    if ((rc = check_length(u, out_len, "output buffer too short"))) return rc;
    uint64_t io[5], oo[5], cnt[5];
    for (int v = 0; v < 5; v++) {
        io[v] = c.v[v].off;
        oo[v] = u.v[v].off;
        cnt[v] = c.v[v].count;
    }
    return copy_vectors(p->curve, in, io, 1, out, oo, 0, cnt, check);
}

int ss_phase1_sizes_of(const ss_phase1_params* p, ss_phase1_sizes* out) { return phase1_sizes(p, out); }

// Phase1::initialization — phase1/src/initialization.rs:12-57: every slot of the accumulator holds the group
// generator (BatchSerializer::init_element, setup-utils/src/io/write.rs:45-55).  The generator is serialized once
// on the device (encode_point) and replicated into the caller's buffer; the 64-byte hash prefix is not touched.
int ss_phase1_initialization(const ss_phase1_params* p, uint8_t* output, size_t output_len, int compressed_output) {
    if (!p || !output) return fail(SS_ERR_INVALID_ARGUMENT, 0, 0, 0, "null argument");
    Phase1Layout L;  // split_mut (buffers.rs:246-288)
    int rc = phase1_layout(p, compressed_output, &L);
    if (rc) return rc;
    const GroupOps* gs[2] = {L.v[0].ops, L.v[1].ops};
    if (p->proving_system != SS_MARLIN && p->proving_system != SS_GROTH16)
        return fail(SS_ERR_INVALID_ARGUMENT, 0, 0, 0, "unknown proving system %d", p->proving_system);
    if ((rc = check_length(L, output_len, "output buffer too short"))) return rc;
    if (!gs[0]->has_generator || !gs[1]->has_generator)
        return fail(SS_ERR_INVALID_ARGUMENT, 0, 0, 0, "the reference's generator constant of %s is not known to this build",
                    gs[0]->has_generator ? gs[1]->name : gs[0]->name);
    if ((rc = ensure_init())) return rc;
    LaneGuard lg;
    if ((rc = lane_acquire(g_devices[0], 4096, &lg.l))) return rc;
    uint8_t gen[2][576];
    for (int g = 0; g < 2; g++) {
        gs[g]->generator(reinterpret_cast<uint32_t*>(lg.l->buf) + g * 256, compressed_output, lg.l->stream);
        CU(cudaGetLastError());
        CU(cudaMemcpyAsync(gen[g], lg.l->buf + g * 1024, compressed_output ? gs[g]->csize : gs[g]->usize,
                           cudaMemcpyDeviceToHost, lg.l->stream));
    }
    CU(cudaStreamSynchronize(lg.l->stream));
    auto fill = [&](uint8_t* dst, const uint8_t* el, uint64_t sz, uint64_t count) {
        if (!count) return;
        memcpy(dst, el, sz);
        for (uint64_t done = 1; done < count;) {  // doubling copies
            const uint64_t k = std::min(done, count - done);
            memcpy(dst + done * sz, dst, k * sz);
            done += k;
        }
    };
    for (const Phase1Layout::Vector& e : L.v) fill(output + e.off, gen[e.group], e.size, e.count);
    return SS_OK;
}

// iter_chunk — phase1/src/helpers/buffers.rs:22-73: the reference's window schedule (windows of
// batch_size elements, consecutive windows overlapping by one).  Host index arithmetic only; the engine
// itself tiles whole vectors, this is exported for callers that keep the reference's loop structure.
int ss_phase1_iter_chunk(const ss_phase1_params* p, uint64_t* starts, uint64_t* ends, size_t max_windows, size_t* count) {
    ss_phase1_sizes z;
    int rc = phase1_sizes(p, &z);
    if (rc) return rc;
    if (!count) return fail(SS_ERR_INVALID_ARGUMENT, 0, 0, 0, "null count");
    if (p->batch_size < 2) return fail(SS_ERR_INVALID_CHUNK, 0, 0, 0, "batch_size must be at least 2");
    const uint64_t upper = p->proving_system == SS_GROTH16 ? z.powers_g1_length : z.powers_length;
    uint64_t lo = 0, hi = upper;
    if (p->contribution_mode == SS_MODE_CHUNKED) {
        lo = p->chunk_index * p->chunk_size;
        hi = std::min<uint64_t>((p->chunk_index + 1) * p->chunk_size, upper);
    }
    const uint64_t step = p->batch_size - 1;
    size_t n = 0;
    auto emit = [&](uint64_t s, uint64_t e) {
        if (n < max_windows && starts && ends) {
            starts[n] = s;
            ends[n] = e;
        }
        n++;
    };
    for (uint64_t i = lo; i < hi; i += step) {
        const uint64_t last = std::min<uint64_t>(i + step, hi) - 1;  // last index of this group
        if (last > i) {
            emit(i, last >= hi - 1 ? last + 1 : last + 2);
        } else if (i >= hi - 1) {
            if (hi == lo + 1) emit(i, i + 1);  // a single trailing element was already covered by the overlap
        } else {
            emit(i, i + 2);
        }
    }
    *count = n;
    if (n > max_windows && starts) return fail(SS_ERR_INVALID_LENGTH, 0, n, max_windows, "window buffer too small");
    return SS_OK;
}

int ss_phase1_computation(const ss_phase1_params* p, const uint8_t* input, size_t input_len, uint8_t* output,
                          size_t output_len, int compressed_input, int compressed_output, int check_input,
                          const uint8_t* tau, const uint8_t* alpha, const uint8_t* beta) {
    return phase1_computation_impl(p, input, input_len, output, output_len, compressed_input, compressed_output,
                                   check_input, tau, alpha, beta, true, nullptr);
}

int ss_phase1_computation_dev(const ss_phase1_params* p, const void* d_input, size_t input_len, void* d_output,
                              size_t output_len, int compressed_input, int compressed_output, int check_input,
                              const uint8_t* tau, const uint8_t* alpha, const uint8_t* beta, void* stream) {
    return phase1_computation_impl(p, static_cast<const uint8_t*>(d_input), input_len, static_cast<uint8_t*>(d_output),
                                   output_len, compressed_input, compressed_output, check_input, tau, alpha, beta,
                                   false, static_cast<cudaStream_t>(stream));
}

// Index-range shard of ONE ceremony (SURVEY.md §8e): every vector of the challenge is cut into `shard_count` equal
// contiguous parts and this call processes part `shard_index` (element i of the vector still gets tau^(first + i)).
// `input` / `output` are the WHOLE challenge / response buffers — typically the same file mapped by every
// process — and only the shard's byte ranges are read and written, the contract the reference's sibling tasks
// already rely on (computation.rs:82-186).  beta_g2 belongs to shard 0.  No inter-process traffic.
int ss_phase1_computation_shard(const ss_phase1_params* p, const uint8_t* input, size_t input_len, uint8_t* output,
                                size_t output_len, int compressed_input, int compressed_output, int check_input,
                                const uint8_t* tau, const uint8_t* alpha, const uint8_t* beta, uint32_t shard_index,
                                uint32_t shard_count) {
    return phase1_computation_impl(p, input, input_len, output, output_len, compressed_input, compressed_output,
                                   check_input, tau, alpha, beta, true, nullptr, shard_index, shard_count);
}

int ss_phase1_computation_shard_dev(const ss_phase1_params* p, const void* d_input, size_t input_len, void* d_output,
                                    size_t output_len, int compressed_input, int compressed_output, int check_input,
                                    const uint8_t* tau, const uint8_t* alpha, const uint8_t* beta, uint32_t shard_index,
                                    uint32_t shard_count, void* stream) {
    return phase1_computation_impl(p, static_cast<const uint8_t*>(d_input), input_len, static_cast<uint8_t*>(d_output),
                                   output_len, compressed_input, compressed_output, check_input, tau, alpha, beta,
                                   false, static_cast<cudaStream_t>(stream), shard_index, shard_count);
}

}  // extern "C"

#include "api_fft.inl"
#include "api_pairing.inl"
#include "api_qap.inl"
