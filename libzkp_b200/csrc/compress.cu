// compress.cu — ark-serialize's compressed form (Compress::Yes) of proofs and keys next to the uncompressed one.
//
// Decoding a compressed point needs a square root (Fq for G1, Fq2 for G2): independent big-integer work per point, run
// here one thread per point (k_decompress).  Compressed keys are decoded on the device in bounded chunks into the
// uncompressed layout in host memory, the device scratch is released, and the bytes go to lzkp_pk_load_ex / lzkp_vk_load:
// every loading path (resident tables or large mode, sharding, validation, the replicas of lzkp_init(n > 1)) is the
// uncompressed one, fed the decoded bytes.  Proofs decode on the caller's stream, so lzkp_proofs_decompress_device
// followed by lzkp_verify_batch_device verifies compressed proofs without a copy through the host.
// Compression is format work (a sign from y per point) and runs on the host for keys and host proofs, on the device for
// device proofs (k_compress_proofs).
#include <algorithm>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "common.h"
#include "point_codec.cuh"

namespace lzkp {
namespace {

constexpr int kThreads = 128;
constexpr size_t kKeyChunk = size_t(1) << 20;          // points per device pass of a key: <= 192 MB of scratch
constexpr size_t kProofChunk = size_t(1) << 20;        // proofs per pass of lzkp_proofs_decompress: 385 MB of scratch

// Proof = A(G1) || B(G2) || C(G1): 256 B uncompressed, 128 B compressed.  A malformed row compresses to 128 bytes of
// 0xFF: coordinates >= q with both flags set, which no reader accepts.
LZ_HD bool compress_proof(const uint8_t *in, uint8_t *out) {
    const bool good = compress_g1(in, out) & compress_g2(in + 64, out + 32) & compress_g1(in + 192, out + 96);
    if (!good) memset(out, 0xFF, 128);
    return good;
}

// One thread per point; rows `in_stride` / `out_stride` bytes apart.  A point that does not decode gets 0xFF over its
// 64 * G output bytes, an encoding every reader - the key loaders and every verifier form - rejects as malformed.
// ok (optional) receives the decision, ANDed with what it holds when ok_and != 0 (the second and third point of a
// proof); bad (optional) counts the points that do not decode.
template <int G>
__global__ void __launch_bounds__(kThreads) k_decompress(const uint8_t *__restrict__ in, size_t in_stride,
                                                         uint8_t *__restrict__ out, size_t out_stride, size_t n,
                                                         uint8_t *__restrict__ ok, int ok_and, uint32_t *__restrict__ bad) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint8_t *o = out + i * out_stride;
    const bool good = G == 1 ? decompress_g1(in + i * in_stride, o) : decompress_g2(in + i * in_stride, o);
    if (!good) memset(o, 0xFF, 64 * G);
    if (ok) ok[i] = (uint8_t)(good && (!ok_and || ok[i]));
    if (!good && bad) atomicAdd(bad, 1u);
}

__global__ void __launch_bounds__(kThreads) k_compress_proofs(const uint8_t *__restrict__ in, uint8_t *__restrict__ out,
                                                              uint8_t *__restrict__ ok, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    ok[i] = compress_proof(in + 256 * i, out + 128 * i) ? 1 : 0;
}

inline unsigned grid_for(size_t n) { return (unsigned)((n + kThreads - 1) / kThreads); }

int enqueue_decompress_proofs(size_t n, const uint8_t *in, uint8_t *out, uint8_t *ok, cudaStream_t st) {
    const unsigned g = grid_for(n);
    LAUNCH(k_decompress<1>, g, kThreads, 0, st, in, 128, out, 256, n, ok, 0, nullptr);              // A
    LAUNCH(k_decompress<2>, g, kThreads, 0, st, in + 32, 128, out + 64, 256, n, ok, 1, nullptr);    // B
    LAUNCH(k_decompress<1>, g, kThreads, 0, st, in + 96, 128, out + 192, 256, n, ok, 1, nullptr);   // C
    CUDA_TRY(cudaGetLastError());
    return LZKP_OK;
}

// ---- key layouts: '1' G1, '2' G2, 'a' Vec<G1>, 'b' Vec<G2> (u64 LE length, then the items)
constexpr char kVkLayout[] = "1222a";                    // alpha, beta, gamma, delta, gamma_abc
constexpr char kPkLayout[] = "1222a11aabaa";             // vk, beta_g1, delta_g1, a, b_g1, b_g2, h, l

struct Seg { int group; size_t in_off, out_off, count; };     // a run of points of one group
struct Plan {
    std::vector<Seg> segs;
    std::vector<std::pair<size_t, size_t>> prefixes;          // (input, output) offsets of the length prefixes
    size_t out_len = 0;
};
// Walks a key of either form; false for a truncated key, a length that overruns the bytes or trailing bytes.
bool plan_key(const uint8_t *b, size_t len, const char *layout, bool compressed_in, Plan &p) {
    const size_t in1 = compressed_in ? 32 : 64, out1 = compressed_in ? 64 : 32;
    size_t ip = 0, op = 0;
    for (const char *c = layout; *c; c++) {
        const size_t g = (*c == '1' || *c == 'a') ? 1 : 2, isz = in1 * g, osz = out1 * g;
        uint64_t cnt = 1;
        if (*c == 'a' || *c == 'b') {
            if (len - ip < 8) return false;
            memcpy(&cnt, b + ip, 8);
            p.prefixes.push_back({ip, op});
            ip += 8;
            op += 8;
        }
        if (cnt > (len - ip) / isz) return false;
        if (cnt) p.segs.push_back({(int)g, ip, op, (size_t)cnt});
        ip += cnt * isz;
        op += cnt * osz;
    }
    if (ip != len) return false;
    p.out_len = op;
    return true;
}

int compress_key(const uint8_t *b, size_t len, const char *layout, const char *what, uint8_t *out, size_t cap,
                 size_t *out_len) {
    if (!b || !out_len) return eng::fail(LZKP_E_INVALID, "null argument");
    Plan p;
    if (!plan_key(b, len, layout, false, p)) return eng::fail(LZKP_E_INVALID, std::string(what) + ": malformed ark-serialize bytes");
    *out_len = p.out_len;
    if (!out) return LZKP_OK;
    if (cap < p.out_len) return eng::fail(LZKP_E_INVALID, std::string(what) + ": output buffer too small");
    for (auto &pr : p.prefixes) memcpy(out + pr.second, b + pr.first, 8);
    for (const Seg &s : p.segs)
        for (size_t k = 0; k < s.count; k++) {
            const uint8_t *src = b + s.in_off + k * 64 * s.group;
            uint8_t *dst = out + s.out_off + k * 32 * s.group;
            if (!(s.group == 1 ? compress_g1(src, dst) : compress_g2(src, dst)))
                return eng::fail(LZKP_E_INVALID, std::string(what) + ": malformed point (non-canonical coordinate or bad flags)");
        }
    return LZKP_OK;
}

// Compressed key bytes -> uncompressed key bytes in `out`, decoded on the device in chunks of kKeyChunk points.  The
// device scratch is released when this returns, before the caller loads the key (pk_load_impl sizes its window tables
// from the free device memory).
int decompress_key(const uint8_t *b, size_t len, const char *layout, const char *what, std::unique_ptr<uint8_t[]> &out,
                   size_t &out_len) {
    Plan p;
    if (!plan_key(b, len, layout, true, p)) return eng::fail(LZKP_E_INVALID, std::string(what) + ": malformed ark-serialize bytes");
    out.reset(new (std::nothrow) uint8_t[p.out_len]);
    if (!out) return eng::fail(LZKP_E_NOMEM, "host allocation failed");
    out_len = p.out_len;
    for (auto &pr : p.prefixes) memcpy(out.get() + pr.second, b + pr.first, 8);
    size_t chunk = 0, g_max = 1;
    for (const Seg &s : p.segs) { chunk = std::max(chunk, std::min(s.count, kKeyChunk)); g_max = std::max<size_t>(g_max, s.group); }
    eng::DBuf d_in, d_out, d_bad;
    TRY(d_in.alloc(std::max<size_t>(chunk, 1) * 32 * g_max));
    TRY(d_out.alloc(std::max<size_t>(chunk, 1) * 64 * g_max));
    TRY(d_bad.alloc(sizeof(uint32_t)));
    CUDA_TRY(cudaMemset(d_bad.p, 0, sizeof(uint32_t)));
    for (const Seg &s : p.segs) {
        const size_t isz = 32 * s.group, osz = 64 * s.group;
        for (size_t off = 0; off < s.count; off += kKeyChunk) {
            const size_t m = std::min(kKeyChunk, s.count - off);
            CUDA_TRY(cudaMemcpy(d_in.p, b + s.in_off + off * isz, m * isz, cudaMemcpyHostToDevice));
            if (s.group == 1) LAUNCH(k_decompress<1>, grid_for(m), kThreads, 0, 0, d_in.as<uint8_t>(), 32, d_out.as<uint8_t>(), 64, m, nullptr, 0, d_bad.as<uint32_t>());
            else LAUNCH(k_decompress<2>, grid_for(m), kThreads, 0, 0, d_in.as<uint8_t>(), 64, d_out.as<uint8_t>(), 128, m, nullptr, 0, d_bad.as<uint32_t>());
            CUDA_TRY(cudaGetLastError());
            CUDA_TRY(cudaMemcpy(out.get() + s.out_off + off * osz, d_out.p, m * osz, cudaMemcpyDeviceToHost));
        }
    }
    uint32_t bad = 0;
    CUDA_TRY(cudaMemcpy(&bad, d_bad.p, sizeof(bad), cudaMemcpyDeviceToHost));
    if (bad) return eng::fail(LZKP_E_INVALID, std::string(what) + ": " + std::to_string(bad) + " compressed point(s) do not decode");
    return LZKP_OK;
}

// Device memory of the calling thread's device (a host pointer would fault in the kernels).
int check_device_buffer(const void *p, const char *what) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return eng::fail(LZKP_E_INVALID, std::string(what) + ": not a CUDA pointer");
    }
    if ((a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) || a.device != eng::current_device())
        return eng::fail(LZKP_E_INVALID, std::string(what) + ": not device memory of the engine's device");
    return LZKP_OK;
}

}  // namespace
}  // namespace lzkp

using namespace lzkp;
using eng::fail;

#pragma GCC visibility push(default)
extern "C" {

int lzkp_pk_load_compressed(const uint8_t *pk_bytes, size_t len, int validate, const lzkp_pk_options *opt, lzkp_pk **out) {
    if (!pk_bytes || !out) return fail(LZKP_E_INVALID, "null argument");
    *out = nullptr;
    TRY(eng::ensure_device());
    std::unique_ptr<uint8_t[]> raw;
    size_t raw_len = 0;
    TRY(decompress_key(pk_bytes, len, kPkLayout, "proving key", raw, raw_len));
    return lzkp_pk_load_ex(raw.get(), raw_len, validate, opt, out);
}

int lzkp_vk_load_compressed(const uint8_t *vk_bytes, size_t len, lzkp_vk **out) {
    if (!vk_bytes || !out) return fail(LZKP_E_INVALID, "null argument");
    *out = nullptr;
    TRY(eng::ensure_device());
    std::unique_ptr<uint8_t[]> raw;
    size_t raw_len = 0;
    TRY(decompress_key(vk_bytes, len, kVkLayout, "verifying key", raw, raw_len));
    return lzkp_vk_load(raw.get(), raw_len, out);
}

int lzkp_pk_compress(const uint8_t *pk_bytes, size_t len, uint8_t *out, size_t cap, size_t *out_len) {
    return compress_key(pk_bytes, len, kPkLayout, "proving key", out, cap, out_len);
}

int lzkp_vk_compress(const uint8_t *vk_bytes, size_t len, uint8_t *out, size_t cap, size_t *out_len) {
    return compress_key(vk_bytes, len, kVkLayout, "verifying key", out, cap, out_len);
}

int lzkp_proofs_compress(size_t n, const uint8_t *proofs, uint8_t *out, uint8_t *ok_out) {
    if (n && (!proofs || !out || !ok_out)) return fail(LZKP_E_INVALID, "null argument");
    for (size_t i = 0; i < n; i++) ok_out[i] = compress_proof(proofs + 256 * i, out + 128 * i) ? 1 : 0;
    return LZKP_OK;
}

int lzkp_proofs_decompress(size_t n, const uint8_t *in, uint8_t *proofs_out, uint8_t *ok_out) {
    if (n && (!in || !proofs_out || !ok_out)) return fail(LZKP_E_INVALID, "null argument");
    TRY(eng::ensure_device());
    if (n == 0) return LZKP_OK;
    const size_t chunk = std::min(n, kProofChunk);
    eng::DBuf d_in, d_out, d_ok;
    TRY(d_in.alloc(chunk * 128));
    TRY(d_out.alloc(chunk * 256));
    TRY(d_ok.alloc(chunk));
    for (size_t off = 0; off < n; off += chunk) {
        const size_t m = std::min(chunk, n - off);
        CUDA_TRY(cudaMemcpy(d_in.p, in + off * 128, m * 128, cudaMemcpyHostToDevice));
        TRY(enqueue_decompress_proofs(m, d_in.as<uint8_t>(), d_out.as<uint8_t>(), d_ok.as<uint8_t>(), 0));
        CUDA_TRY(cudaMemcpy(proofs_out + off * 256, d_out.p, m * 256, cudaMemcpyDeviceToHost));
        CUDA_TRY(cudaMemcpy(ok_out + off, d_ok.p, m, cudaMemcpyDeviceToHost));
    }
    return LZKP_OK;
}

int lzkp_proofs_compress_device(size_t n, const void *d_in, void *d_out, void *d_ok, void *stream) {
    if (n && (!d_in || !d_out || !d_ok)) return fail(LZKP_E_INVALID, "null argument");
    TRY(eng::ensure_device());
    if (n == 0) return LZKP_OK;
    TRY(check_device_buffer(d_in, "proofs"));
    TRY(check_device_buffer(d_out, "compressed proofs"));
    TRY(check_device_buffer(d_ok, "ok"));
    LAUNCH(k_compress_proofs, grid_for(n), kThreads, 0, (cudaStream_t)stream, (const uint8_t *)d_in, (uint8_t *)d_out,
           (uint8_t *)d_ok, n);
    CUDA_TRY(cudaGetLastError());
    return LZKP_OK;
}

int lzkp_proofs_decompress_device(size_t n, const void *d_in, void *d_proofs_out, void *d_ok, void *stream) {
    if (n && (!d_in || !d_proofs_out || !d_ok)) return fail(LZKP_E_INVALID, "null argument");
    TRY(eng::ensure_device());
    if (n == 0) return LZKP_OK;
    TRY(check_device_buffer(d_in, "compressed proofs"));
    TRY(check_device_buffer(d_proofs_out, "proofs"));
    TRY(check_device_buffer(d_ok, "ok"));
    return enqueue_decompress_proofs(n, (const uint8_t *)d_in, (uint8_t *)d_proofs_out, (uint8_t *)d_ok,
                                     (cudaStream_t)stream);
}

}  // extern "C"
#pragma GCC visibility pop
