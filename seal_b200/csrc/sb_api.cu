// seal_b200/csrc/sb_api.cu -- the extern "C" boundary declared in include/seal_b200.h.
// Exceptions never cross it: they are mapped to status codes the way the reference's C layer maps them to HRESULTs
// (native/src/seal/c/defines.h:72-96) and the message is kept in a thread-local string.
#include "../../include/seal_b200.h"
#include "sb_engine.cuh"
#include <random>
#include <algorithm>
#include <cctype>
#include <cstdio>
#include <cstring>
#include <new>
#include <thread>

using namespace sb;

static thread_local std::string g_last_error;

struct sb200_context
{
    std::unique_ptr<Context> c;
};
struct sb200_public_key
{
    PublicKey k;
    ~sb200_public_key()
    {
        if (k.d_key && k.ctx)
        {
            cudaSetDevice(k.ctx->device);
            cudaFree(k.d_key);
        }
    }
};
struct sb200_secret_key
{
    SecretKey k;
    // the reference keeps SecretKey data in a clear-on-destruction pool (secretkey.h:51-60): wipe before the memory goes back
    // to the allocator
    ~sb200_secret_key()
    {
        if (k.d_pow && k.ctx)
        {
            cudaSetDevice(k.ctx->device);
            cudaMemset(k.d_pow, 0, k.powers * k.ctx->k * k.ctx->n * sizeof(u64));
            cudaDeviceSynchronize();
        }
        cudaFree(k.d_pow);
    }
};
struct sb200_kswitch_key
{
    KSwitchKey k;
    ~sb200_kswitch_key()
    {
        if (k.ctx)
            cudaSetDevice(k.ctx->device);
        cudaFree(k.d_key);
        cudaFree(k.d_key32);
    }
};

#define SB_TRY try {
#define SB_CATCH                                   \
    }                                              \
    catch (const std::invalid_argument &e)         \
    {                                              \
        g_last_error = e.what();                   \
        return SB200_E_INVALID_ARG;                \
    }                                              \
    catch (const std::out_of_range &e)             \
    {                                              \
        g_last_error = e.what();                   \
        return SB200_E_OUT_OF_RANGE;               \
    }                                              \
    catch (const std::logic_error &e)              \
    {                                              \
        g_last_error = e.what();                   \
        return SB200_E_LOGIC;                      \
    }                                              \
    catch (const std::bad_alloc &e)                \
    {                                              \
        g_last_error = e.what();                   \
        return SB200_E_NOMEM;                      \
    }                                              \
    catch (const std::exception &e)                \
    {                                              \
        g_last_error = e.what();                   \
        return SB200_E_CUDA;                       \
    }

#define SB_NEED(p)                                      \
    if (!(p))                                           \
    {                                                   \
        g_last_error = "null pointer: " #p;             \
        return SB200_E_POINTER;                         \
    }

extern "C" {

const char *sb200_last_error(void)
{
    return g_last_error.c_str();
}

int sb200_context_create(int scheme, size_t n, const uint64_t *coeff_modulus, size_t k, uint64_t plain_modulus, int device,
                         sb200_context **out)
{
    SB_NEED(coeff_modulus);
    SB_NEED(out);
    SB_TRY
    auto h = std::make_unique<sb200_context>();
    h->c = make_context(scheme, n, reinterpret_cast<const u64 *>(coeff_modulus), k, plain_modulus, device);
    *out = h.release();
    return SB200_OK;
    SB_CATCH
}

int sb200_context_destroy(sb200_context *ctx)
{
    SB_NEED(ctx);
    delete ctx;
    return SB200_OK;
}

int sb200_coeff_modulus_create(size_t n, const int *bit_sizes, size_t k, uint64_t *out)
{
    SB_NEED(bit_sizes);
    SB_NEED(out);
    SB_TRY
    if (n < 2 || (n & (n - 1)) || n > 131072)
        throw std::invalid_argument("poly_modulus_degree is invalid");
    for (size_t i = 0; i < k; i++)
        if (bit_sizes[i] < 2 || bit_sizes[i] > 60)
            throw std::invalid_argument("bit_sizes is invalid");
    auto v = sbh::coeff_modulus_create(n, std::vector<int>(bit_sizes, bit_sizes + k));
    for (size_t i = 0; i < k; i++)
        out[i] = v[i];
    return SB200_OK;
    SB_CATCH
}

int sb200_get_ntt_tables(const sb200_context *ctx, size_t i, uint64_t *root, uint64_t *rp_op, uint64_t *rp_quo, uint64_t *irp_op,
                         uint64_t *inv_n)
{
    SB_NEED(ctx);
    SB_TRY
    const Context &c = *ctx->c;
    if (i >= c.k)
        throw std::out_of_range("prime_index");
    const auto &t = c.tabs[i];
    if (root)
        *root = t.root;
    if (inv_n)
        *inv_n = t.inv_n.w;
    for (size_t j = 0; j < c.n; j++)
    {
        if (rp_op)
            rp_op[j] = t.root_powers[j].w;
        if (rp_quo)
            rp_quo[j] = t.root_powers[j].wq;
        if (irp_op)
            irp_op[j] = t.inv_root_powers[j].w;
    }
    return SB200_OK;
    SB_CATCH
}

int sb200_get_base_bsk(const sb200_context *ctx, size_t L, uint64_t *out, size_t capacity, size_t *count)
{
    SB_NEED(ctx);
    SB_NEED(out);
    SB_NEED(count);
    SB_TRY
    Context &c = *ctx->c;
    if (c.scheme != SB200_SCHEME_BFV)
        throw std::logic_error("BEHZ base exists for BFV contexts only");
    const auto &b = behz_host(c, L);
    if (b.nBsk > capacity)
        throw std::out_of_range("capacity");
    for (size_t i = 0; i < b.nBsk; i++)
        out[i] = b.Bsk[i];
    *count = b.nBsk;
    return SB200_OK;
    SB_CATCH
}

uint32_t sb200_galois_elt_from_step(const sb200_context *ctx, int step)
{
    if (!ctx)
        return 0;
    try
    {
        return sbh::galois_elt_from_step(ctx->c->n, step);
    }
    catch (const std::exception &e)
    {
        g_last_error = e.what();
        return 0;
    }
}

unsigned long long sb200_launch_count(const sb200_context *ctx)
{
    return ctx ? ctx->c->stats.launches : 0;
}

size_t sb200_device_bytes(const sb200_context *ctx)
{
    return ctx ? ctx->c->table_bytes + ctx->c->scratch_bytes + ctx->c->aux_bytes : 0;
}

int sb200_context_set_limit(sb200_context *ctx, int which, size_t value)
{
    SB_NEED(ctx);
    SB_TRY
    Context &c = *ctx->c;
    std::lock_guard<std::mutex> lock(c.mu);
    switch (which)
    {
    case SB200_LIMIT_SCRATCH_BYTES: c.scratch_budget = std::max<size_t>(value, size_t(1) << 20); break;
    case SB200_LIMIT_KS_CHUNK: c.ks_chunk_max = value; break;
    case SB200_LIMIT_HOST_STAGE_BYTES: c.host_stage_bytes = std::max<size_t>(value, size_t(1) << 16); break;
    case SB200_LIMIT_KS_ALGORITHM:
        if (value > 2)
            throw std::invalid_argument("unknown key-switching algorithm");
        c.ks_algo = static_cast<int>(value);
        break;
    default: throw std::invalid_argument("unknown limit");
    }
    return SB200_OK;
    SB_CATCH
}

// ---- device-resident slabs / staging memory ----
int sb200_device_malloc(sb200_context *ctx, size_t bytes, uint64_t **d_out)
{
    SB_NEED(ctx);
    SB_NEED(d_out);
    SB_TRY
    Context &c = *ctx->c;
    cuda_check(cudaSetDevice(c.device), "cudaSetDevice");
    void *p = nullptr;
    cudaError_t e = cudaMalloc(&p, std::max<size_t>(bytes, 8));
    if (e == cudaErrorMemoryAllocation)
    {
        cudaGetLastError();
        throw std::bad_alloc();
    }
    cuda_check(e, "cudaMalloc(slab)");
    *d_out = static_cast<uint64_t *>(p);
    return SB200_OK;
    SB_CATCH
}
int sb200_device_free(sb200_context *ctx, uint64_t *d_ptr)
{
    SB_NEED(ctx);
    SB_TRY
    cuda_check(cudaSetDevice(ctx->c->device), "cudaSetDevice");
    cuda_check(cudaFree(d_ptr), "cudaFree(slab)");
    return SB200_OK;
    SB_CATCH
}
int sb200_host_malloc(sb200_context *ctx, size_t bytes, void **h_out)
{
    SB_NEED(ctx);
    SB_NEED(h_out);
    SB_TRY
    cuda_check(cudaSetDevice(ctx->c->device), "cudaSetDevice");
    void *p = nullptr;
    cudaError_t e = cudaHostAlloc(&p, std::max<size_t>(bytes, 8), cudaHostAllocDefault);
    if (e == cudaErrorMemoryAllocation)
    {
        cudaGetLastError();
        throw std::bad_alloc();
    }
    cuda_check(e, "cudaHostAlloc");
    *h_out = p;
    return SB200_OK;
    SB_CATCH
}
int sb200_host_free(sb200_context *ctx, void *h_ptr)
{
    SB_NEED(ctx);
    SB_TRY
    cuda_check(cudaFreeHost(h_ptr), "cudaFreeHost");
    return SB200_OK;
    SB_CATCH
}
static int copy_(sb200_context *ctx, void *dst, const void *src, size_t bytes, cudaMemcpyKind kind, void *stream)
{
    SB_NEED(ctx);
    SB_NEED(dst);
    SB_NEED(src);
    SB_TRY
    cuda_check(cudaSetDevice(ctx->c->device), "cudaSetDevice");
    cuda_check(cudaMemcpyAsync(dst, src, bytes, kind, static_cast<cudaStream_t>(stream)), "cudaMemcpyAsync");
    return SB200_OK;
    SB_CATCH
}
int sb200_memcpy_h2d(sb200_context *ctx, uint64_t *d_dst, const void *h_src, size_t bytes, void *stream)
{
    return copy_(ctx, d_dst, h_src, bytes, cudaMemcpyHostToDevice, stream);
}
int sb200_memcpy_d2h(sb200_context *ctx, void *h_dst, const uint64_t *d_src, size_t bytes, void *stream)
{
    return copy_(ctx, h_dst, d_src, bytes, cudaMemcpyDeviceToHost, stream);
}
int sb200_memcpy_d2d(sb200_context *ctx, uint64_t *d_dst, const uint64_t *d_src, size_t bytes, void *stream)
{
    return copy_(ctx, d_dst, d_src, bytes, cudaMemcpyDeviceToDevice, stream);
}
int sb200_memcpy_d2d_2d(sb200_context *ctx, uint64_t *d_dst, size_t dst_pitch, const uint64_t *d_src, size_t src_pitch, size_t row_bytes,
                        size_t rows, void *stream)
{
    SB_NEED(ctx);
    SB_NEED(d_dst);
    SB_NEED(d_src);
    SB_TRY
    cuda_check(cudaSetDevice(ctx->c->device), "cudaSetDevice");
    cuda_check(cudaMemcpy2DAsync(d_dst, dst_pitch, d_src, src_pitch, row_bytes, rows, cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream)),
               "cudaMemcpy2DAsync");
    return SB200_OK;
    SB_CATCH
}
int sb200_stream_synchronize(sb200_context *ctx, void *stream)
{
    SB_NEED(ctx);
    SB_TRY
    cuda_check(cudaSetDevice(ctx->c->device), "cudaSetDevice");
    cuda_check(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)), "cudaStreamSynchronize");
    return SB200_OK;
    SB_CATCH
}
} // extern "C"
namespace
{
    // copies rows [r0, r1) between the caller's objects and a contiguous page-locked buffer on a few host threads (one thread
    // moves ~10 GB/s, a Gen5 x16 link 50+ GB/s)
    void rows_copy(bool gather, uint8_t *stage, const uint64_t *const *rows, size_t row_bytes, size_t r0, size_t r1)
    {
        const size_t cnt = r1 - r0;
        const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
        const size_t nt = std::max<size_t>(1, std::min<size_t>({ 8, hw / 2 ? hw / 2 : 1, cnt * row_bytes / (size_t(4) << 20) + 1 }));
        auto work = [&](size_t t) {
            // split by bytes so that few large rows still spread over all threads
            const size_t total = cnt * row_bytes, b0 = total * t / nt, b1 = total * (t + 1) / nt;
            for (size_t off = b0; off < b1;)
            {
                const size_t r = off / row_bytes, in = off % row_bytes, len = std::min(row_bytes - in, b1 - off);
                uint8_t *user = reinterpret_cast<uint8_t *>(const_cast<uint64_t *>(rows[r0 + r])) + in;
                if (gather)
                    std::memcpy(stage + off, user, len);
                else
                    std::memcpy(user, stage + off, len);
                off += len;
            }
        };
        if (nt == 1)
            return work(0);
        std::vector<std::thread> th;
        for (size_t t = 1; t < nt; t++)
            th.emplace_back(work, t);
        work(0);
        for (auto &x : th)
            x.join();
    }
    void ensure_lane(Context &c, IoArena::Lane &ln, size_t bytes)
    {
        if (!ln.st)
        {
            cuda_check(cudaStreamCreateWithFlags(&ln.st, cudaStreamNonBlocking), "cudaStreamCreate");
            cuda_check(cudaEventCreateWithFlags(&ln.order, cudaEventDisableTiming), "cudaEventCreate");
            for (int i = 0; i < 2; i++)
                cuda_check(cudaEventCreateWithFlags(&ln.ev[i], cudaEventDisableTiming), "cudaEventCreate");
        }
        if (ln.cap >= bytes)
            return;
        for (int i = 0; i < 2; i++)
        {
            cudaFreeHost(ln.pin[i]);
            ln.pin[i] = nullptr;
        }
        ln.cap = 0;
        for (int i = 0; i < 2; i++)
            cuda_check(cudaHostAlloc(&ln.pin[i], bytes, cudaHostAllocDefault), "cudaHostAlloc(staging)");
        ln.cap = bytes;
    }
    // The copies run on the lane's own non-blocking stream: they overlap kernels of other batches.  Ordering with the caller's
    // work: a download first waits for everything the legacy default stream has been given so far (the batch operations of the
    // C++ shim enqueue there); an upload returns when the data has arrived, so whatever the caller enqueues next sees it.
    void rows_transfer(Context &c, bool upload, uint64_t *dev, const uint64_t *const *rows, size_t row_bytes, size_t count)
    {
        if (!count || !row_bytes)
            return;
        IoArena::Lane &ln = c.io.lane[upload ? 0 : 1];
        std::lock_guard<std::mutex> lock(ln.mu);
        cuda_check(cudaSetDevice(c.device), "cudaSetDevice");
        const size_t per = std::max<size_t>(1, (size_t(128) << 20) / row_bytes), stage_bytes = std::min(per, count) * row_bytes;
        ensure_lane(c, ln, stage_bytes);
        cudaStream_t st = ln.st;
        if (!upload)
        {
            cuda_check(cudaEventRecord(ln.order, nullptr), "record");
            cuda_check(cudaStreamWaitEvent(st, ln.order, 0), "wait");
        }
        uint8_t *d = reinterpret_cast<uint8_t *>(dev);
        size_t i = 0, pend[2] = { 0, 0 }, pend_n[2] = { 0, 0 };
        bool used[2] = { false, false };
        for (size_t r0 = 0; r0 < count; r0 += per, i++)
        {
            const size_t r1 = std::min(count, r0 + per);
            const int slot = static_cast<int>(i & 1);
            uint8_t *stage = static_cast<uint8_t *>(ln.pin[slot]);
            if (used[slot])
            {
                cuda_check(cudaEventSynchronize(ln.ev[slot]), "cudaEventSynchronize");
                if (!upload)
                    rows_copy(false, stage, rows, row_bytes, pend[slot], pend[slot] + pend_n[slot]);
            }
            if (upload)
            {
                rows_copy(true, stage, rows, row_bytes, r0, r1);
                cuda_check(cudaMemcpyAsync(d + r0 * row_bytes, stage, (r1 - r0) * row_bytes, cudaMemcpyHostToDevice, st), "H2D");
            }
            else
                cuda_check(cudaMemcpyAsync(stage, d + r0 * row_bytes, (r1 - r0) * row_bytes, cudaMemcpyDeviceToHost, st), "D2H");
            cuda_check(cudaEventRecord(ln.ev[slot], st), "record");
            used[slot] = true, pend[slot] = r0, pend_n[slot] = r1 - r0;
        }
        // drain in submission order
        for (size_t j = (i >= 2 ? i - 2 : 0); j < i; j++)
        {
            const int slot = static_cast<int>(j & 1);
            cuda_check(cudaEventSynchronize(ln.ev[slot]), "cudaEventSynchronize");
            if (!upload)
                rows_copy(false, static_cast<uint8_t *>(ln.pin[slot]), rows, row_bytes, pend[slot], pend[slot] + pend_n[slot]);
        }
    }
} // namespace
extern "C" {
int sb200_upload_rows(sb200_context *ctx, uint64_t *d_dst, const uint64_t *const *h_rows, size_t row_bytes, size_t count)
{
    SB_NEED(d_dst);
    SB_NEED(h_rows);
    SB_TRY
    SB_NEED(ctx);
    rows_transfer(*ctx->c, true, d_dst, h_rows, row_bytes, count);
    return SB200_OK;
    SB_CATCH
}
int sb200_download_rows(sb200_context *ctx, uint64_t *const *h_rows, const uint64_t *d_src, size_t row_bytes, size_t count)
{
    SB_NEED(d_src);
    SB_NEED(h_rows);
    SB_TRY
    SB_NEED(ctx);
    rows_transfer(*ctx->c, false, const_cast<uint64_t *>(d_src), h_rows, row_bytes, count);
    return SB200_OK;
    SB_CATCH
}
int sb200_device_index(const sb200_context *ctx)
{
    return ctx ? ctx->c->device : -1;
}
int sb200_device_numa_node(const sb200_context *ctx)
{
    if (!ctx)
        return -1;
    char bus[32] = { 0 };
    if (cudaDeviceGetPCIBusId(bus, sizeof(bus), ctx->c->device) != cudaSuccess)
        return -1;
    for (char *p = bus; *p; p++)
        *p = static_cast<char>(std::tolower(*p));
    std::string path = std::string("/sys/bus/pci/devices/") + bus + "/numa_node";
    int node = -1;
    if (FILE *f = std::fopen(path.c_str(), "r"))
    {
        if (std::fscanf(f, "%d", &node) != 1)
            node = -1;
        std::fclose(f);
    }
    return node;
}
size_t sb200_keyswitch_chunk(const sb200_context *ctx, size_t L, size_t batch, int fused)
{
    return ctx ? sb::keyswitch_chunk(*ctx->c, L, batch, fused != 0) : 0;
}

int sb200_profile_enable(sb200_context *ctx, int on)
{
    SB_NEED(ctx);
    std::lock_guard<std::mutex> lock(ctx->c->mu);
    ctx->c->stats.profiling = (on != 0);
    return SB200_OK;
}

int sb200_profile_reset(sb200_context *ctx)
{
    SB_NEED(ctx);
    std::lock_guard<std::mutex> lock(ctx->c->mu);
    cudaSetDevice(ctx->c->device);
    cudaDeviceSynchronize();
    ctx->c->stats.clear();
    return SB200_OK;
}

int sb200_profile_read(sb200_context *ctx, size_t index, char *name, size_t name_capacity, double *total_ms,
                       unsigned long long *launches, double *algorithmic_bytes)
{
    return sb200_profile_read_work(ctx, index, name, name_capacity, total_ms, launches, algorithmic_bytes, nullptr, nullptr);
}

int sb200_selftest_ksint_info(sb200_context *ctx, int *count, uint32_t *primes)
{
    SB_NEED(ctx);
    SB_NEED(count);
    SB_NEED(primes);
    const KsInt &d = ctx->c->ksint;
    *count = d.ready ? d.prm.S : 0;
    for (int t = 0; t < *count; t++)
        primes[t] = d.prm.p[t];
    return SB200_OK;
}

int sb200_selftest_ksint_forward(sb200_context *ctx, const uint64_t *h_rows, size_t rows, uint32_t *h_out)
{
    SB_NEED(ctx);
    SB_NEED(h_rows);
    SB_NEED(h_out);
    SB_TRY
    Context &c = *ctx->c;
    std::lock_guard<std::mutex> lock(c.mu);
    cuda_check(cudaSetDevice(c.device), "cudaSetDevice");
    ksint_selftest_transform(c, false, reinterpret_cast<const u64 *>(h_rows), rows, h_out);
    return SB200_OK;
    SB_CATCH
}

int sb200_selftest_ksint_inverse(sb200_context *ctx, uint32_t *h_data, size_t rows)
{
    SB_NEED(ctx);
    SB_NEED(h_data);
    SB_TRY
    Context &c = *ctx->c;
    std::lock_guard<std::mutex> lock(c.mu);
    cuda_check(cudaSetDevice(c.device), "cudaSetDevice");
    ksint_selftest_transform(c, true, nullptr, rows, h_data);
    return SB200_OK;
    SB_CATCH
}

int sb200_selftest_rate(sb200_context *ctx, int kind, double *warp_ops_per_second)
{
    SB_NEED(warp_ops_per_second);
    SB_NEED(ctx);
    SB_TRY
    Context &c = *ctx->c;
    std::lock_guard<std::mutex> lock(c.mu);
    cuda_check(cudaSetDevice(c.device), "cudaSetDevice");
    *warp_ops_per_second = kind >= 10 ? ksint_selftest_rate(c, kind - 10, nullptr) : selftest_rate(c, kind, nullptr);
    return SB200_OK;
    SB_CATCH
}

int sb200_profile_read_work(sb200_context *ctx, size_t index, char *name, size_t name_capacity, double *total_ms,
                            unsigned long long *launches, double *algorithmic_bytes, double *butterflies, double *macs)
{
    return sb200_profile_read_work32(ctx, index, name, name_capacity, total_ms, launches, algorithmic_bytes, butterflies, macs, nullptr, nullptr);
}

int sb200_profile_read_work32(sb200_context *ctx, size_t index, char *name, size_t name_capacity, double *total_ms,
                              unsigned long long *launches, double *algorithmic_bytes, double *butterflies, double *macs,
                              double *butterflies32, double *macs32)
{
    SB_NEED(ctx);
    SB_NEED(name);
    SB_NEED(total_ms);
    SB_NEED(launches);
    SB_NEED(algorithmic_bytes);
    SB_TRY
    Context &c = *ctx->c;
    std::lock_guard<std::mutex> lock(c.mu);
    cuda_check(cudaSetDevice(c.device), "cudaSetDevice");
    cuda_check(cudaDeviceSynchronize(), "synchronize");
    // aggregate by (name, pass) in first-seen order
    struct Agg
    {
        std::string name;
        double ms = 0, bytes = 0, bflys = 0, macs = 0, bflys32 = 0, macs32 = 0;
        unsigned long long n = 0;
    };
    std::vector<Agg> aggs;
    static const char *suffix[] = { "", ":col", ":local" };
    for (auto &r : c.stats.recs)
    {
        std::string nm = std::string(r.name) + suffix[r.pass];
        float ms = 0;
        cuda_check(cudaEventElapsedTime(&ms, r.e0, r.e1), "cudaEventElapsedTime");
        auto it = std::find_if(aggs.begin(), aggs.end(), [&](const Agg &a) { return a.name == nm; });
        if (it == aggs.end())
        {
            aggs.push_back(Agg{ nm });
            it = aggs.end() - 1;
        }
        it->ms += ms, it->bytes += r.bytes, it->bflys += r.bflys, it->macs += r.macs, it->bflys32 += r.bflys32, it->macs32 += r.macs32, it->n++;
    }
    if (index >= aggs.size())
        throw std::out_of_range("profile index");
    std::snprintf(name, name_capacity, "%s", aggs[index].name.c_str());
    *total_ms = aggs[index].ms;
    *launches = aggs[index].n;
    *algorithmic_bytes = aggs[index].bytes;
    if (butterflies)
        *butterflies = aggs[index].bflys;
    if (macs)
        *macs = aggs[index].macs;
    if (butterflies32)
        *butterflies32 = aggs[index].bflys32;
    if (macs32)
        *macs32 = aggs[index].macs32;
    return SB200_OK;
    SB_CATCH
}

int sb200_kswitch_key_create(sb200_context *ctx, const uint64_t *h_key, size_t digits, sb200_kswitch_key **out)
{
    SB_NEED(ctx);
    SB_NEED(h_key);
    SB_NEED(out);
    SB_TRY
    Context &c = *ctx->c;
    if (c.k < 2)
        throw std::logic_error("keyswitching is not supported by the context");
    if (digits < 1 || digits > c.k - 1)
        throw std::invalid_argument("kswitch key has an invalid number of digits");
    auto h = std::make_unique<sb200_kswitch_key>();
    size_t bytes = digits * 2 * c.k * c.n * sizeof(u64);
    std::lock_guard<std::mutex> lock(c.mu);
    cuda_check(cudaSetDevice(c.device), "cudaSetDevice");
    cuda_check(cudaMalloc(reinterpret_cast<void **>(&h->k.d_key), bytes), "cudaMalloc(key)");
    cuda_check(cudaMemcpy(h->k.d_key, h_key, bytes, cudaMemcpyHostToDevice), "upload key");
    h->k.ctx = &c;
    h->k.digits = digits;
    // is_data_valid_for (valcheck.cpp:412-456): every word below its modulus -- the fused key-switch kernel relies on it to
    // keep its 128-bit sums in range
    if (!op_residues_in_range(c, c.k, digits * 2 * c.k, h->k.d_key, nullptr))
        throw std::invalid_argument("kswitch key data is not valid for encryption parameters");
    ksint_prepare_key(c, h->k, nullptr);
    *out = h.release();
    return SB200_OK;
    SB_CATCH
}

int sb200_kswitch_key_load(sb200_context *ctx, const uint8_t *stream, size_t len, size_t index, sb200_kswitch_key **out)
{
    SB_NEED(ctx);
    SB_NEED(stream);
    SB_NEED(out);
    SB_TRY
    Context &c = *ctx->c;
    if (c.k < 2)
        throw std::logic_error("keyswitching is not supported by the context");
    sbw::KSwitchEntry e;
    std::vector<uint8_t> plain; // KSwitchKeys saved with compr_mode_type::zlib: inflate the object, then parse as usual
    // bound: a GaloisKeys object holds at most 2 log2(n) + 1 < 64 keys of k-1 digits, plus one size word per slot
    if (sbw::inflate_stream(stream, len, 64 * (c.k - 1) * sbw::save_size(2 * c.k * c.n) + 16 * c.n + 4096, plain))
        stream = plain.data(), len = plain.size();
    sbw::inspect_kswitch(stream, len, index, e);
    // is_valid_for(KSwitchKeys): keys live at the key level of this context (valcheck.cpp, kswitchkeys.cpp:149-153)
    if (e.n != c.n || e.L != c.k || std::memcmp(e.parms_id, c.parms_ids[c.k - 1].data(), sizeof(e.parms_id)) != 0)
        throw std::logic_error("KSwitchKeys data is invalid");
    const size_t digits = e.offsets.size();
    // is_valid_for(KSwitchKeys) (valcheck.cpp:292-323): one public key per decomposition prime, i.e. exactly k-1 digits
    if (digits != c.k - 1)
        throw std::logic_error("KSwitchKeys data is invalid");
    auto h = std::make_unique<sb200_kswitch_key>();
    const size_t row = 2 * c.k * c.n * sizeof(u64);
    std::lock_guard<std::mutex> lock(c.mu);
    cuda_check(cudaSetDevice(c.device), "cudaSetDevice");
    cuda_check(cudaMalloc(reinterpret_cast<void **>(&h->k.d_key), digits * row), "cudaMalloc(key)");
    for (size_t j = 0; j < digits; j++)
        cuda_check(cudaMemcpy(reinterpret_cast<uint8_t *>(h->k.d_key) + j * row, stream + e.offsets[j], row, cudaMemcpyHostToDevice), "upload key");
    h->k.ctx = &c;
    h->k.digits = digits;
    if (!op_residues_in_range(c, c.k, digits * 2 * c.k, h->k.d_key, nullptr)) // KSwitchKeys::load ends in is_valid_for (kswitchkeys.cpp:149-153)
        throw std::logic_error("KSwitchKeys data is invalid");
    ksint_prepare_key(c, h->k, nullptr);
    *out = h.release();
    return SB200_OK;
    SB_CATCH
}

int sb200_kswitch_key_destroy(sb200_kswitch_key *key)
{
    SB_NEED(key);
    delete key;
    return SB200_OK;
}

#define SB_ENTER(ctx)                                      \
    SB_NEED(ctx);                                          \
    Context &c = *ctx->c;                                  \
    std::lock_guard<std::mutex> lock(c.mu);                \
    cuda_check(cudaSetDevice(c.device), "cudaSetDevice");

// The scratch arenas of a context are shared by all of its calls.  Calls on one stream are ordered by the stream; a call on a
// different stream than the previous one first waits for that one's work (one event record per call, no host synchronisation).
namespace
{
    struct StreamOrder
    {
        Context &c;
        cudaStream_t st;
        StreamOrder(Context &ctx, cudaStream_t stream) : c(ctx), st(stream)
        {
            if (c.order_valid && c.order_stream != st)
                cuda_check(cudaStreamWaitEvent(st, c.order_event, 0), "cudaStreamWaitEvent(order)");
        }
        ~StreamOrder()
        {
            if (!c.order_event && cudaEventCreateWithFlags(&c.order_event, cudaEventDisableTiming) != cudaSuccess)
                return;
            if (cudaEventRecord(c.order_event, st) == cudaSuccess)
                c.order_stream = st, c.order_valid = true;
        }
    };
} // namespace
#define SB_ENTER_STREAM(ctx, stream) \
    SB_ENTER(ctx)                    \
    StreamOrder order_(c, static_cast<cudaStream_t>(stream));

static void check_level(const Context &c, size_t L, size_t batch)
{
    if (L < 1 || L > c.k)
        throw std::invalid_argument("encrypted is not valid for encryption parameters");
    if (batch == 0)
        throw std::invalid_argument("batch must be positive");
}

static void check_size(size_t size)
{
    if (size < 1 || size > 16) // SEAL_CIPHERTEXT_SIZE_MAX (util/defines.h)
        throw std::invalid_argument("invalid ciphertext size");
}

// SB_NEED for an argument the device and host entry points name differently: the message keeps each entry point's name
#define SB_NEED_AS(p, name)                                    \
    if (!(p))                                                  \
    {                                                          \
        g_last_error = std::string("null pointer: ") + (name); \
        return SB200_E_POINTER;                                \
    }
} // extern "C"

// ---- evaluator operations ------------------------------------------------------------------------------------------
// Each operation is written once, as a template over where its data lives: its null checks, then (under the context's lock)
// its argument checks, which return the words per ciphertext of its slabs, and its driver call on ciphertexts
// [first, first + B).  OnDevice runs it on the caller's device slabs and stream; OnHost runs it on host buffers through HostPipe.
namespace
{
    struct Slabs
    {
        size_t wa, wb, wo; // words per ciphertext of input a, input b (0 = none), output (0 = in place in a)
    };

    // The batch is cut into chunks that flow through a 3-stage pipeline on three streams: H2D copy of chunk i+1 | kernels
    // of chunk i | D2H copy of chunk i-1, double-buffered device staging owned by the context (PCIe is full duplex, so with
    // pinned host buffers both copy directions overlap each other and the compute).  Pageable host memory works too, the
    // copies then serialise inside the driver.
    struct HostPipe
    {
        Context &c;
        cudaStream_t s_in, s_comp, s_out;
        cudaEvent_t ev_in[2], ev_comp[2], ev_out[2];
        explicit HostPipe(Context &ctx) : c(ctx)
        {
            IoArena &io = c.io;
            if (!io.ready)
            {
                for (auto *s : { &io.s_in, &io.s_comp, &io.s_out })
                    cuda_check(cudaStreamCreateWithFlags(s, cudaStreamNonBlocking), "cudaStreamCreate");
                for (int i = 0; i < 2; i++)
                    for (auto *e : { &io.ev_in[i], &io.ev_comp[i], &io.ev_out[i] })
                        cuda_check(cudaEventCreateWithFlags(e, cudaEventDisableTiming), "cudaEventCreate");
                io.ready = true;
            }
            s_in = io.s_in, s_comp = io.s_comp, s_out = io.s_out;
            for (int i = 0; i < 2; i++)
                ev_in[i] = io.ev_in[i], ev_comp[i] = io.ev_comp[i], ev_out[i] = io.ev_out[i];
        }
        u64 *buffer(int slot, int which, size_t words)
        {
            IoArena &io = c.io;
            size_t &cap = io.cap[slot][which];
            if (words > cap)
            {
                cuda_check(cudaDeviceSynchronize(), "sync before io growth");
                cudaFree(io.buf[slot][which]);
                io.buf[slot][which] = nullptr;
                cap = 0;
                cuda_check(cudaMalloc(reinterpret_cast<void **>(&io.buf[slot][which]), words * sizeof(u64)), "cudaMalloc(io)");
                cap = words;
            }
            return io.buf[slot][which];
        }
        // op(c, first, B, da, db, dout, stream) runs the operation on ciphertexts [first, first + B) of the batch
        template <class F>
        void run(size_t batch, const Slabs &s, const uint64_t *ha, const uint64_t *hb, uint64_t *ho, F &&op)
        {
            const size_t wa = s.wa, wb = s.wb, wo = s.wo, wout = wo ? wo : wa;
            const size_t per_ct = (wa + wb + wo) * sizeof(u64);
            size_t chunk = std::max<size_t>(1, std::min<size_t>(batch, c.host_stage_bytes / std::max<size_t>(per_ct, 1)));
            if (chunk >= batch && batch >= 4)
                chunk = (batch + 1) / 2; // at least two chunks so the copies overlap the kernels
            if (chunk < batch)
            {
                // A chunk's D2H copy is not ordered before the H2D copies of later chunks.  So with several chunks the output may
                // overlap an input only exactly in place with an output no larger than that input: chunk i's output then lies
                // inside the input of chunks <= i, which are on the device already.  (With one chunk every H2D copy precedes the
                // kernels and they precede the D2H copy, so any overlap is safe.)
                const uintptr_t o0 = reinterpret_cast<uintptr_t>(ho), o1 = o0 + batch * wout * sizeof(u64);
                auto unsafe = [&](const uint64_t *hx, size_t wx) {
                    const uintptr_t x0 = reinterpret_cast<uintptr_t>(hx), x1 = x0 + batch * wx * sizeof(u64);
                    return x0 < o1 && o0 < x1 && !(hx == ho && wout <= wx);
                };
                if (unsafe(ha, wa) || (wb && unsafe(hb, wb)))
                    throw std::invalid_argument("the output buffer overlaps an input buffer: a batch of several staging chunks may only run "
                                                "exactly in place, with an output no larger than the input");
            }
            StreamOrder order(c, s_comp); // the operation's kernels (and the scratch arenas they use) run on s_comp
            // size all staging (and let the op grow its scratch) before the pipeline starts: growth synchronises the device
            for (int slot = 0; slot < 2; slot++)
            {
                buffer(slot, 0, chunk * wa);
                if (wb)
                    buffer(slot, 1, chunk * wb);
                if (wo)
                    buffer(slot, 2, chunk * wo);
            }
            size_t i = 0;
            for (size_t b0 = 0; b0 < batch; b0 += chunk, i++)
            {
                const size_t B = std::min(chunk, batch - b0);
                const int slot = static_cast<int>(i & 1);
                u64 *da = buffer(slot, 0, B * wa), *db = wb ? buffer(slot, 1, B * wb) : nullptr, *dout = wo ? buffer(slot, 2, B * wo) : da;
                if (i >= 2)
                {
                    // inputs of this slot are free once its previous kernels finished (and, in place, once copied out)
                    cuda_check(cudaStreamWaitEvent(s_in, wo ? ev_comp[slot] : ev_out[slot], 0), "wait");
                }
                cuda_check(cudaMemcpyAsync(da, ha + b0 * wa, B * wa * sizeof(u64), cudaMemcpyHostToDevice, s_in), "H2D");
                if (wb)
                    cuda_check(cudaMemcpyAsync(db, hb + b0 * wb, B * wb * sizeof(u64), cudaMemcpyHostToDevice, s_in), "H2D");
                cuda_check(cudaEventRecord(ev_in[slot], s_in), "record");
                cuda_check(cudaStreamWaitEvent(s_comp, ev_in[slot], 0), "wait");
                if (i >= 2 && wo)
                    cuda_check(cudaStreamWaitEvent(s_comp, ev_out[slot], 0), "wait"); // output staging of this slot drained
                op(c, b0, B, da, db, dout, s_comp);
                cuda_check(cudaEventRecord(ev_comp[slot], s_comp), "record");
                cuda_check(cudaStreamWaitEvent(s_out, ev_comp[slot], 0), "wait");
                cuda_check(cudaMemcpyAsync(ho + b0 * wout, dout, B * wout * sizeof(u64), cudaMemcpyDeviceToHost, s_out), "D2H");
                cuda_check(cudaEventRecord(ev_out[slot], s_out), "record");
            }
            cuda_check(cudaStreamSynchronize(s_out), "synchronize");
            cuda_check(cudaStreamSynchronize(s_comp), "synchronize");
        }
    };

    // Device entry points: the checks, then the driver on the whole batch on the caller's stream.  secret: the call handled
    // secret data, which must not stay behind in the scratch arenas.
    struct OnDevice
    {
        static constexpr bool device = true;
        void *stream;
        template <class Check, class Drive>
        int run(sb200_context *ctx, size_t batch, const uint64_t *a, const uint64_t *b, uint64_t *out, Check &&check, Drive &&drive,
                bool secret = false) const
        {
            SB_TRY
            SB_ENTER_STREAM(ctx, stream)
            check(c);
            const auto st = static_cast<cudaStream_t>(stream);
            drive(c, size_t(0), batch, reinterpret_cast<const u64 *>(a), reinterpret_cast<const u64 *>(b), reinterpret_cast<u64 *>(out), st);
            if (secret)
                c.wipe_scratch(st); // the decryption phases (decryptor.cpp:106-109 keeps them in a clearing pool)
            return SB200_OK;
            SB_CATCH
        }
    };

    // Host-buffer entry points: the checks, then the pipeline over the batch; nothing is copied before every check has passed.
    struct OnHost
    {
        static constexpr bool device = false;
        template <class Check, class Drive>
        int run(sb200_context *ctx, size_t batch, const uint64_t *a, const uint64_t *b, uint64_t *out, Check &&check, Drive &&drive,
                bool secret = false) const
        {
            SB_TRY
            SB_ENTER(ctx)
            const Slabs s = check(c);
            HostPipe(c).run(batch, s, a, b, out, drive);
            if (secret)
            {
                // phases and plaintexts do not stay behind in the arenas (the reference decrypts inside a clear-on-destruction pool)
                c.wipe_scratch(c.io.s_comp);
                for (int slot = 0; slot < 2; slot++)
                    if (c.io.buf[slot][2])
                        cuda_check(cudaMemsetAsync(c.io.buf[slot][2], 0, c.io.cap[slot][2] * sizeof(u64), c.io.s_comp), "wipe staging");
                cuda_check(cudaStreamSynchronize(c.io.s_comp), "synchronize");
            }
            return SB200_OK;
            SB_CATCH
        }
    };

    template <class Where>
    int ntt_(Where w, sb200_context *ctx, bool inverse, size_t L, size_t size, size_t batch, uint64_t *data)
    {
        SB_NEED_AS(data, Where::device ? "d" : "h");
        return w.run(
            ctx, batch, data, nullptr, data,
            [&](Context &c) {
                check_level(c, L, batch);
                return Slabs{ size * L * c.n, 0, 0 };
            },
            [&](Context &c, size_t, size_t B, const u64 *, const u64 *, u64 *dout, cudaStream_t st) { op_ntt(c, inverse, L, size, B, dout, st); });
    }

    // Evaluator::multiply of size_a x size_b ciphertexts: CKKS and BGV share the NTT-form tensor (evaluator.cpp:569-708, :710-841),
    // BFV runs BEHZ.  Both drivers take their size-2 kernels for sizes (2, 2) and square with their own kernel when a == b.
    void tensor(Context &c, size_t L, size_t size_a, size_t size_b, size_t B, const u64 *a, const u64 *b, u64 *out, cudaStream_t st)
    {
        if (c.scheme != SB200_SCHEME_BFV)
            op_ckks_multiply(c, L, size_a, size_b, B, a, b, out, st);
        else
            op_bfv_multiply(c, L, size_a, size_b, B, a, b, out, st);
    }

    template <class Where>
    int multiply_(Where w, sb200_context *ctx, size_t L, size_t batch, const uint64_t *a, const uint64_t *b, uint64_t *out3)
    {
        SB_NEED(a);
        SB_NEED(b);
        SB_NEED(out3);
        return w.run(
            ctx, batch, a, b, out3,
            [&](Context &c) {
                check_level(c, L, batch);
                return Slabs{ 2 * L * c.n, 2 * L * c.n, 3 * L * c.n };
            },
            [&](Context &c, size_t, size_t B, const u64 *da, const u64 *db, u64 *dout, cudaStream_t st) { tensor(c, L, 2, 2, B, da, db, dout, st); });
    }

    template <class Where>
    int multiply_sized_(Where w, sb200_context *ctx, size_t L, size_t size_a, size_t size_b, size_t batch, const uint64_t *a, const uint64_t *b,
                        uint64_t *out)
    {
        SB_NEED(a);
        SB_NEED(b);
        SB_NEED(out);
        return w.run(
            ctx, batch, a, b, out,
            [&](Context &c) {
                check_level(c, L, batch);
                if (Where::device && (out == a || out == b))
                    throw std::invalid_argument("multiply: the output slab must not alias an input slab");
                check_sizes(size_a, size_b);
                return Slabs{ size_a * L * c.n, size_b * L * c.n, (size_a + size_b - 1) * L * c.n };
            },
            [&](Context &c, size_t, size_t B, const u64 *da, const u64 *db, u64 *dout, cudaStream_t st) {
                tensor(c, L, size_a, size_b, B, da, db, dout, st);
            });
    }

    template <class Where>
    int square_(Where w, sb200_context *ctx, size_t L, size_t batch, const uint64_t *a, uint64_t *out3)
    {
        SB_NEED(a);
        SB_NEED(out3);
        return w.run(
            ctx, batch, a, nullptr, out3,
            [&](Context &c) {
                check_level(c, L, batch);
                return Slabs{ 2 * L * c.n, 0, 3 * L * c.n }; // one operand crosses the bus
            },
            [&](Context &c, size_t, size_t B, const u64 *da, const u64 *, u64 *dout, cudaStream_t st) { tensor(c, L, 2, 2, B, da, da, dout, st); });
    }

    // mode 0: add, 1: sub, 2: negate (no b)
    template <class Where>
    int linear_(Where w, sb200_context *ctx, int mode, size_t L, size_t size, size_t batch, const uint64_t *a, const uint64_t *b, uint64_t *out)
    {
        SB_NEED(a);
        SB_NEED(out);
        if (mode != 2)
            SB_NEED(b);
        return w.run(
            ctx, batch, a, b, out,
            [&](Context &c) {
                check_level(c, L, batch);
                const size_t words = size * L * c.n;
                return Slabs{ words, mode == 2 ? 0 : words, words };
            },
            [&](Context &c, size_t, size_t B, const u64 *da, const u64 *db, u64 *dout, cudaStream_t st) {
                op_linear(c, mode, L, size, B, da, db, dout, st);
            });
    }

    template <class Where>
    int multiply_plain_(Where w, sb200_context *ctx, size_t L, size_t size, size_t batch, const uint64_t *a, const uint64_t *plain, uint64_t *out)
    {
        SB_NEED(a);
        SB_NEED(plain);
        SB_NEED(out);
        return w.run(
            ctx, batch, a, plain, out,
            [&](Context &c) {
                check_level(c, L, batch);
                return Slabs{ size * L * c.n, L * c.n, size * L * c.n };
            },
            [&](Context &c, size_t, size_t B, const u64 *da, const u64 *db, u64 *dout, cudaStream_t st) {
                op_multiply_plain(c, L, size, B, da, db, dout, st);
            });
    }

    template <class Where>
    int plain_to_ntt_(Where w, sb200_context *ctx, size_t L, size_t batch, const uint64_t *plain, uint64_t *out)
    {
        SB_NEED(plain);
        SB_NEED(out);
        return w.run(
            ctx, batch, plain, nullptr, out,
            [&](Context &c) {
                check_level(c, L, batch);
                return Slabs{ c.n, 0, L * c.n };
            },
            [&](Context &c, size_t, size_t B, const u64 *da, const u64 *, u64 *dout, cudaStream_t st) { op_plain_to_ntt(c, L, B, da, nullptr, dout, st); });
    }

    template <class Where>
    int multiply_plain_coeff_(Where w, sb200_context *ctx, size_t L, size_t size, size_t batch, int ct_is_ntt, const uint64_t *a,
                              const uint64_t *plain, uint64_t *out)
    {
        SB_NEED(a);
        SB_NEED(plain);
        SB_NEED(out);
        return w.run(
            ctx, batch, a, plain, out,
            [&](Context &c) {
                check_level(c, L, batch);
                return Slabs{ size * L * c.n, c.n, size * L * c.n };
            },
            [&](Context &c, size_t, size_t B, const u64 *da, const u64 *db, u64 *dout, cudaStream_t st) {
                op_multiply_plain_coeff(c, L, size, B, ct_is_ntt != 0, da, db, dout, st);
            });
    }

    template <class Where>
    int add_plain_coeff_(Where w, sb200_context *ctx, size_t L, size_t size, size_t batch, int subtract, const uint64_t *a, const uint64_t *plain,
                         const uint64_t *h_correction_factors, uint64_t *out)
    {
        SB_NEED(a);
        SB_NEED(plain);
        SB_NEED(out);
        const u64 *h_cf = reinterpret_cast<const u64 *>(h_correction_factors);
        return w.run(
            ctx, batch, a, plain, out,
            [&](Context &c) {
                check_level(c, L, batch);
                return Slabs{ size * L * c.n, c.n, size * L * c.n };
            },
            [&](Context &c, size_t first, size_t B, const u64 *da, const u64 *db, u64 *dout, cudaStream_t st) {
                op_add_plain_coeff(c, L, size, B, subtract != 0, da, db, h_cf ? h_cf + first : nullptr, dout, st);
            });
    }

    template <class Where>
    int batch_codec_(Where w, sb200_context *ctx, bool decode, size_t batch, const uint64_t *in, uint64_t *out)
    {
        SB_NEED(in);
        SB_NEED(out);
        return w.run(
            ctx, batch, in, nullptr, out,
            [&](Context &c) {
                if (batch == 0)
                    throw std::invalid_argument("batch must be positive");
                return Slabs{ c.n, 0, c.n };
            },
            [&](Context &c, size_t, size_t B, const u64 *da, const u64 *, u64 *dout, cudaStream_t st) {
                if (decode)
                    op_batch_decode(c, B, da, dout, st);
                else
                    op_batch_encode(c, B, da, dout, st);
            });
    }

    template <class Where>
    int relinearize_(Where w, sb200_context *ctx, size_t L, size_t batch, const uint64_t *in3, const sb200_kswitch_key *key, uint64_t *out2)
    {
        SB_NEED(in3);
        SB_NEED(key);
        SB_NEED(out2);
        return w.run(
            ctx, batch, in3, nullptr, out2,
            [&](Context &c) {
                check_level(c, L, batch);
                if (Where::device && in3 == out2)
                    throw std::invalid_argument("relinearize: input and output slabs must not alias (different layouts)");
                return Slabs{ 3 * L * c.n, 0, 2 * L * c.n };
            },
            [&](Context &c, size_t, size_t B, const u64 *da, const u64 *, u64 *dout, cudaStream_t st) { op_relinearize(c, L, B, da, key->k, dout, st); });
    }

    template <class Where>
    int multiply_relinearize_(Where w, sb200_context *ctx, size_t L, size_t batch, const uint64_t *a, const uint64_t *b, const sb200_kswitch_key *key,
                              uint64_t *out2)
    {
        SB_NEED(a);
        SB_NEED(b);
        SB_NEED(key);
        SB_NEED(out2);
        return w.run(
            ctx, batch, a, b, out2,
            [&](Context &c) {
                check_level(c, L, batch);
                return Slabs{ 2 * L * c.n, 2 * L * c.n, 2 * L * c.n };
            },
            [&](Context &c, size_t, size_t B, const u64 *da, const u64 *db, u64 *dout, cudaStream_t st) {
                op_multiply_relinearize(c, L, B, da, db, key->k, dout, st);
            });
    }

    template <class Where>
    int relinearize_sized_(Where w, sb200_context *ctx, size_t L, size_t size, size_t batch, const uint64_t *in, const sb200_kswitch_key *key,
                           uint64_t *out)
    {
        SB_NEED(in);
        SB_NEED(key);
        SB_NEED(out);
        return w.run(
            ctx, batch, in, nullptr, out,
            [&](Context &c) {
                check_level(c, L, batch);
                if (Where::device && in == out)
                    throw std::invalid_argument("relinearize: input and output slabs must not alias");
                if (size < 3 || size > 16) // a polynomial to switch and (c_0, c_1); SEAL_CIPHERTEXT_SIZE_MAX
                    throw std::invalid_argument("invalid ciphertext size");
                return Slabs{ size * L * c.n, 0, size * L * c.n };
            },
            [&](Context &c, size_t, size_t B, const u64 *da, const u64 *, u64 *dout, cudaStream_t st) {
                op_relinearize_sized(c, L, size, B, da, key->k, dout, st);
            });
    }

    // rescale: CKKS only (evaluator.cpp:1533); the scheme is checked before the end of the chain, as op_rescale does
    template <class Where>
    int modswitch_(Where w, sb200_context *ctx, bool rescale, size_t L, size_t size, size_t batch, const uint64_t *in, uint64_t *out)
    {
        SB_NEED_AS(in, Where::device ? "in" : "in2");
        SB_NEED_AS(out, Where::device ? "out" : "out2");
        return w.run(
            ctx, batch, in, nullptr, out,
            [&](Context &c) {
                check_level(c, L, batch);
                check_size(size);
                if (Where::device && in == out)
                    throw std::invalid_argument(rescale ? "rescale_to_next: input and output slabs must not alias (different layouts)"
                                                        : "mod_switch_to_next: input and output slabs must not alias (different layouts)");
                if (rescale && c.scheme != SB200_SCHEME_CKKS)
                    throw std::invalid_argument("unsupported operation for scheme type");
                if (L < 2)
                    throw std::invalid_argument("end of modulus switching chain reached");
                return Slabs{ size * L * c.n, 0, size * (L - 1) * c.n };
            },
            [&](Context &c, size_t, size_t B, const u64 *da, const u64 *, u64 *dout, cudaStream_t st) {
                if (rescale)
                    op_rescale(c, L, B * size, da, dout, st);
                else
                    op_mod_switch(c, L, B * size, da, dout, st);
            });
    }

    template <class Where>
    int apply_galois_(Where w, sb200_context *ctx, size_t L, size_t batch, const uint64_t *in2, uint32_t elt, const sb200_kswitch_key *key,
                      uint64_t *out2)
    {
        SB_NEED(in2);
        SB_NEED(key);
        SB_NEED(out2);
        return w.run(
            ctx, batch, in2, nullptr, out2,
            [&](Context &c) {
                check_level(c, L, batch);
                return Slabs{ 2 * L * c.n, 0, 2 * L * c.n };
            },
            [&](Context &c, size_t, size_t B, const u64 *da, const u64 *, u64 *dout, cudaStream_t st) {
                op_apply_galois(c, L, B, da, elt, key->k, dout, st);
            });
    }

    // Decryptor::decrypt (decryptor.cpp:62-197)
    template <class Where>
    int decrypt_(Where w, sb200_context *ctx, sb200_secret_key *key, size_t L, size_t size, size_t batch, const uint64_t *ct,
                 const uint64_t *h_correction_factors, uint64_t *plain)
    {
        SB_NEED(key);
        SB_NEED(ct);
        SB_NEED(plain);
        const u64 *h_cf = reinterpret_cast<const u64 *>(h_correction_factors);
        return w.run(
            ctx, batch, ct, nullptr, plain,
            [&](Context &c) {
                check_level(c, L, batch);
                return Slabs{ size * L * c.n, 0, c.scheme == SB200_SCHEME_CKKS ? L * c.n : c.n };
            },
            [&](Context &c, size_t first, size_t B, const u64 *da, const u64 *, u64 *dout, cudaStream_t st) {
                op_decrypt(c, key->k, L, size, B, da, h_cf ? h_cf + first : nullptr, dout, st);
            },
            true);
    }
} // namespace

extern "C" {

int sb200_ntt_forward(sb200_context *ctx, size_t L, size_t size, size_t batch, uint64_t *d, void *stream)
{
    return ntt_(OnDevice{ stream }, ctx, false, L, size, batch, d);
}
int sb200_ntt_forward_host(sb200_context *ctx, size_t L, size_t size, size_t batch, uint64_t *h)
{
    return ntt_(OnHost{}, ctx, false, L, size, batch, h);
}
int sb200_ntt_inverse(sb200_context *ctx, size_t L, size_t size, size_t batch, uint64_t *d, void *stream)
{
    return ntt_(OnDevice{ stream }, ctx, true, L, size, batch, d);
}
int sb200_ntt_inverse_host(sb200_context *ctx, size_t L, size_t size, size_t batch, uint64_t *h)
{
    return ntt_(OnHost{}, ctx, true, L, size, batch, h);
}

int sb200_multiply(sb200_context *ctx, size_t L, size_t batch, const uint64_t *a, const uint64_t *b, uint64_t *out3, void *stream)
{
    return multiply_(OnDevice{ stream }, ctx, L, batch, a, b, out3);
}
int sb200_multiply_host(sb200_context *ctx, size_t L, size_t batch, const uint64_t *a, const uint64_t *b, uint64_t *out3)
{
    return multiply_(OnHost{}, ctx, L, batch, a, b, out3);
}

int sb200_multiply_sized(sb200_context *ctx, size_t L, size_t size_a, size_t size_b, size_t batch, const uint64_t *a, const uint64_t *b,
                         uint64_t *out, void *stream)
{
    return multiply_sized_(OnDevice{ stream }, ctx, L, size_a, size_b, batch, a, b, out);
}
int sb200_multiply_sized_host(sb200_context *ctx, size_t L, size_t size_a, size_t size_b, size_t batch, const uint64_t *a, const uint64_t *b,
                              uint64_t *out)
{
    return multiply_sized_(OnHost{}, ctx, L, size_a, size_b, batch, a, b, out);
}

int sb200_square(sb200_context *ctx, size_t L, size_t batch, const uint64_t *a, uint64_t *out3, void *stream)
{
    return square_(OnDevice{ stream }, ctx, L, batch, a, out3);
}
int sb200_square_host(sb200_context *ctx, size_t L, size_t batch, const uint64_t *a, uint64_t *out3)
{
    return square_(OnHost{}, ctx, L, batch, a, out3);
}

int sb200_add(sb200_context *ctx, size_t L, size_t size, size_t batch, const uint64_t *a, const uint64_t *b, uint64_t *out, void *stream)
{
    return linear_(OnDevice{ stream }, ctx, 0, L, size, batch, a, b, out);
}
int sb200_add_host(sb200_context *ctx, size_t L, size_t size, size_t batch, const uint64_t *a, const uint64_t *b, uint64_t *out)
{
    return linear_(OnHost{}, ctx, 0, L, size, batch, a, b, out);
}
int sb200_sub(sb200_context *ctx, size_t L, size_t size, size_t batch, const uint64_t *a, const uint64_t *b, uint64_t *out, void *stream)
{
    return linear_(OnDevice{ stream }, ctx, 1, L, size, batch, a, b, out);
}
int sb200_sub_host(sb200_context *ctx, size_t L, size_t size, size_t batch, const uint64_t *a, const uint64_t *b, uint64_t *out)
{
    return linear_(OnHost{}, ctx, 1, L, size, batch, a, b, out);
}
int sb200_negate(sb200_context *ctx, size_t L, size_t size, size_t batch, const uint64_t *a, uint64_t *out, void *stream)
{
    return linear_(OnDevice{ stream }, ctx, 2, L, size, batch, a, nullptr, out);
}
int sb200_negate_host(sb200_context *ctx, size_t L, size_t size, size_t batch, const uint64_t *a, uint64_t *out)
{
    return linear_(OnHost{}, ctx, 2, L, size, batch, a, nullptr, out);
}

int sb200_multiply_plain(sb200_context *ctx, size_t L, size_t size, size_t batch, const uint64_t *a, const uint64_t *plain, uint64_t *out,
                         void *stream)
{
    return multiply_plain_(OnDevice{ stream }, ctx, L, size, batch, a, plain, out);
}
int sb200_multiply_plain_host(sb200_context *ctx, size_t L, size_t size, size_t batch, const uint64_t *a, const uint64_t *plain, uint64_t *out)
{
    return multiply_plain_(OnHost{}, ctx, L, size, batch, a, plain, out);
}

int sb200_plain_to_ntt(sb200_context *ctx, size_t L, size_t batch, const uint64_t *plain, uint64_t *out, void *stream)
{
    return plain_to_ntt_(OnDevice{ stream }, ctx, L, batch, plain, out);
}
int sb200_plain_to_ntt_host(sb200_context *ctx, size_t L, size_t batch, const uint64_t *plain, uint64_t *out)
{
    return plain_to_ntt_(OnHost{}, ctx, L, batch, plain, out);
}

int sb200_multiply_plain_coeff(sb200_context *ctx, size_t L, size_t size, size_t batch, int ct_is_ntt, const uint64_t *a, const uint64_t *plain,
                               uint64_t *out, void *stream)
{
    return multiply_plain_coeff_(OnDevice{ stream }, ctx, L, size, batch, ct_is_ntt, a, plain, out);
}
int sb200_multiply_plain_coeff_host(sb200_context *ctx, size_t L, size_t size, size_t batch, int ct_is_ntt, const uint64_t *a,
                                    const uint64_t *plain, uint64_t *out)
{
    return multiply_plain_coeff_(OnHost{}, ctx, L, size, batch, ct_is_ntt, a, plain, out);
}

int sb200_add_plain_coeff(sb200_context *ctx, size_t L, size_t size, size_t batch, int subtract, const uint64_t *a, const uint64_t *plain,
                          const uint64_t *h_correction_factors, uint64_t *out, void *stream)
{
    return add_plain_coeff_(OnDevice{ stream }, ctx, L, size, batch, subtract, a, plain, h_correction_factors, out);
}
int sb200_add_plain_coeff_host(sb200_context *ctx, size_t L, size_t size, size_t batch, int subtract, const uint64_t *a, const uint64_t *plain,
                               const uint64_t *h_correction_factors, uint64_t *out)
{
    return add_plain_coeff_(OnHost{}, ctx, L, size, batch, subtract, a, plain, h_correction_factors, out);
}

int sb200_batch_encode(sb200_context *ctx, size_t batch, const uint64_t *values, uint64_t *plain, void *stream)
{
    return batch_codec_(OnDevice{ stream }, ctx, false, batch, values, plain);
}
int sb200_batch_encode_host(sb200_context *ctx, size_t batch, const uint64_t *values, uint64_t *plain)
{
    return batch_codec_(OnHost{}, ctx, false, batch, values, plain);
}
int sb200_batch_decode(sb200_context *ctx, size_t batch, const uint64_t *plain, uint64_t *values, void *stream)
{
    return batch_codec_(OnDevice{ stream }, ctx, true, batch, plain, values);
}
int sb200_batch_decode_host(sb200_context *ctx, size_t batch, const uint64_t *plain, uint64_t *values)
{
    return batch_codec_(OnHost{}, ctx, true, batch, plain, values);
}

int sb200_relinearize(sb200_context *ctx, size_t L, size_t batch, const uint64_t *in3, const sb200_kswitch_key *key, uint64_t *out2,
                      void *stream)
{
    return relinearize_(OnDevice{ stream }, ctx, L, batch, in3, key, out2);
}
int sb200_relinearize_host(sb200_context *ctx, size_t L, size_t batch, const uint64_t *in3, const sb200_kswitch_key *key, uint64_t *out2)
{
    return relinearize_(OnHost{}, ctx, L, batch, in3, key, out2);
}

int sb200_multiply_relinearize(sb200_context *ctx, size_t L, size_t batch, const uint64_t *a, const uint64_t *b,
                               const sb200_kswitch_key *key, uint64_t *out2, void *stream)
{
    return multiply_relinearize_(OnDevice{ stream }, ctx, L, batch, a, b, key, out2);
}
int sb200_multiply_relinearize_host(sb200_context *ctx, size_t L, size_t batch, const uint64_t *a, const uint64_t *b,
                                    const sb200_kswitch_key *key, uint64_t *out2)
{
    return multiply_relinearize_(OnHost{}, ctx, L, batch, a, b, key, out2);
}

int sb200_relinearize_sized(sb200_context *ctx, size_t L, size_t size, size_t batch, const uint64_t *in, const sb200_kswitch_key *key,
                            uint64_t *out, void *stream)
{
    return relinearize_sized_(OnDevice{ stream }, ctx, L, size, batch, in, key, out);
}
int sb200_relinearize_sized_host(sb200_context *ctx, size_t L, size_t size, size_t batch, const uint64_t *in, const sb200_kswitch_key *key,
                                 uint64_t *out)
{
    return relinearize_sized_(OnHost{}, ctx, L, size, batch, in, key, out);
}

int sb200_rescale_to_next(sb200_context *ctx, size_t L, size_t batch, const uint64_t *in2, uint64_t *out2, void *stream)
{
    return modswitch_(OnDevice{ stream }, ctx, true, L, 2, batch, in2, out2);
}
int sb200_rescale_to_next_host(sb200_context *ctx, size_t L, size_t batch, const uint64_t *in2, uint64_t *out2)
{
    return modswitch_(OnHost{}, ctx, true, L, 2, batch, in2, out2);
}
int sb200_rescale_to_next_sized(sb200_context *ctx, size_t L, size_t size, size_t batch, const uint64_t *in, uint64_t *out, void *stream)
{
    return modswitch_(OnDevice{ stream }, ctx, true, L, size, batch, in, out);
}
int sb200_rescale_to_next_sized_host(sb200_context *ctx, size_t L, size_t size, size_t batch, const uint64_t *in, uint64_t *out)
{
    return modswitch_(OnHost{}, ctx, true, L, size, batch, in, out);
}
int sb200_mod_switch_to_next(sb200_context *ctx, size_t L, size_t batch, const uint64_t *in2, uint64_t *out2, void *stream)
{
    return modswitch_(OnDevice{ stream }, ctx, false, L, 2, batch, in2, out2);
}
int sb200_mod_switch_to_next_host(sb200_context *ctx, size_t L, size_t batch, const uint64_t *in2, uint64_t *out2)
{
    return modswitch_(OnHost{}, ctx, false, L, 2, batch, in2, out2);
}
int sb200_mod_switch_to_next_sized(sb200_context *ctx, size_t L, size_t size, size_t batch, const uint64_t *in, uint64_t *out, void *stream)
{
    return modswitch_(OnDevice{ stream }, ctx, false, L, size, batch, in, out);
}
int sb200_mod_switch_to_next_sized_host(sb200_context *ctx, size_t L, size_t size, size_t batch, const uint64_t *in, uint64_t *out)
{
    return modswitch_(OnHost{}, ctx, false, L, size, batch, in, out);
}

int sb200_apply_galois(sb200_context *ctx, size_t L, size_t batch, const uint64_t *in2, uint32_t elt, const sb200_kswitch_key *key,
                       uint64_t *out2, void *stream)
{
    return apply_galois_(OnDevice{ stream }, ctx, L, batch, in2, elt, key, out2);
}
int sb200_apply_galois_host(sb200_context *ctx, size_t L, size_t batch, const uint64_t *in2, uint32_t elt, const sb200_kswitch_key *key,
                            uint64_t *out2)
{
    return apply_galois_(OnHost{}, ctx, L, batch, in2, elt, key, out2);
}

int sb200_decrypt(sb200_context *ctx, sb200_secret_key *key, size_t L, size_t size, size_t batch, const uint64_t *ct,
                  const uint64_t *h_correction_factors, uint64_t *plain, void *stream)
{
    return decrypt_(OnDevice{ stream }, ctx, key, L, size, batch, ct, h_correction_factors, plain);
}
int sb200_decrypt_host(sb200_context *ctx, sb200_secret_key *key, size_t L, size_t size, size_t batch, const uint64_t *ct,
                       const uint64_t *h_correction_factors, uint64_t *plain)
{
    return decrypt_(OnHost{}, ctx, key, L, size, batch, ct, h_correction_factors, plain);
}

// ---- wire format (SURVEY 8f rank 3): Ciphertext::save / load, compr_mode none, between byte streams and device slabs ----
int sb200_get_parms_id(const sb200_context *ctx, size_t L, uint64_t out[4])
{
    SB_NEED(ctx);
    SB_NEED(out);
    SB_TRY
    const Context &c = *ctx->c;
    if (L < 1 || L > c.k)
        throw std::out_of_range("L");
    for (int i = 0; i < 4; i++)
        out[i] = c.parms_ids[L - 1][i];
    return SB200_OK;
    SB_CATCH
}

int sb200_ciphertext_inspect(const uint8_t *stream, size_t len, sb200_ct_info *info)
{
    SB_NEED(stream);
    SB_NEED(info);
    SB_TRY
    std::vector<uint8_t> plain;
    // a compressed object is inflated first (bounded by the largest ciphertext the format allows: 16 x 256 x 131072 words)
    if (sbw::inflate_stream(stream, len, sbw::save_size(size_t(16) * 256 * 131072) + 128, plain))
    {
        sbw::inspect(plain.data(), plain.size(), *info);
        uint64_t total = 0;
        std::memcpy(&total, stream + 8, sizeof(total)); // SEALHeader::size of the stream as given
        info->stream_bytes = total;
        info->compr_mode = 1;
    }
    else
        sbw::inspect(stream, len, *info);
    return SB200_OK;
    SB_CATCH
}

size_t sb200_ciphertext_save_size(const sb200_context *ctx, size_t L, size_t size)
{
    return ctx ? sbw::save_size(size * L * ctx->c->n) : 0;
}

int sb200_ciphertext_load(sb200_context *ctx, size_t batch, const uint8_t *const *streams, const size_t *lens, size_t L, size_t size,
                          int validate, uint64_t *d_out, sb200_ct_info *infos, void *stream)
{
    SB_NEED(streams);
    SB_NEED(lens);
    SB_NEED(d_out);
    SB_TRY
    SB_ENTER_STREAM(ctx, stream)
    check_level(c, L, batch);
    auto st = static_cast<cudaStream_t>(stream);
    const size_t words = size * L * c.n;
    std::vector<u64> seeds;            // seeded members: 8 words each
    std::vector<long long> seed_dst;   // word offset of their second polynomial in d_out
    for (size_t b = 0; b < batch; b++)
    {
        sb200_ct_info info;
        std::vector<uint8_t> plain; // a zlib-compressed member is inflated on the host (bounded by the shape asked for)
        const uint8_t *src = streams[b];
        if (!src)
            throw std::invalid_argument("in cannot be null");
        if (sbw::inflate_stream(src, lens[b], sbw::save_size(words) + 128, plain))
        {
            sbw::inspect(plain.data(), plain.size(), info);
            src = plain.data();
            info.compr_mode = 1;
        }
        else
            sbw::inspect(src, lens[b], info);
        if (info.seeded == 2)
            throw std::logic_error("unsupported prng_type"); // shake256 streams stay with the reference (ciphertext.cpp:124-128)
        // is_metadata_valid_for (ciphertext.cpp:299-302): the stream must belong to this context at the level asked for
        if (info.poly_modulus_degree != c.n || info.coeff_modulus_size != L || info.size != size ||
            std::memcmp(info.parms_id, c.parms_ids[L - 1].data(), sizeof(info.parms_id)) != 0)
            throw std::logic_error("ciphertext data is invalid");
        if (infos)
            infos[b] = info;
        // (pageable source: the call returns once the bytes have left the buffer, so `plain` may go out of scope)
        cuda_check(cudaMemcpyAsync(d_out + b * words, src + info.data_offset, info.data_words * sizeof(u64), cudaMemcpyHostToDevice, st), "H2D");
        if (info.seeded)
        {
            u64 sd[8];
            std::memcpy(sd, src + info.seed_offset, sizeof(sd));
            seeds.insert(seeds.end(), sd, sd + 8);
            seed_dst.push_back(static_cast<long long>(b * words + L * c.n));
        }
    }
    if (!seed_dst.empty())
        op_expand_seeded(c, L, seed_dst.size(), seeds.data(), seed_dst.data(), reinterpret_cast<u64 *>(d_out), st); // Ciphertext::expand_seed
    if (validate && !op_residues_in_range(c, L, batch * size * L, reinterpret_cast<const u64 *>(d_out), st))
        throw std::logic_error("ciphertext data is invalid"); // Ciphertext::load -> is_valid_for (ciphertext.h:640-655)
    return SB200_OK;
    SB_CATCH
}

int sb200_ciphertext_save(sb200_context *ctx, size_t batch, size_t L, size_t size, const uint64_t *d_in, const sb200_ct_info *meta,
                          uint8_t *const *outs, size_t capacity, void *stream)
{
    SB_NEED(d_in);
    SB_NEED(meta);
    SB_NEED(outs);
    SB_TRY
    SB_ENTER_STREAM(ctx, stream)
    check_level(c, L, batch);
    auto st = static_cast<cudaStream_t>(stream);
    const size_t words = size * L * c.n;
    if (size < 2 || size > 16)
        throw std::invalid_argument("invalid size");
    if (capacity < sbw::save_size(words))
        throw std::invalid_argument("insufficient size"); // Serialization::Save into a too small buffer
    for (size_t b = 0; b < batch; b++)
    {
        if (!outs[b])
            throw std::invalid_argument("out cannot be null");
        sb200_ct_info info = meta[b];
        std::memcpy(info.parms_id, c.parms_ids[L - 1].data(), sizeof(info.parms_id));
        info.size = size, info.poly_modulus_degree = c.n, info.coeff_modulus_size = L, info.data_words = words;
        sbw::write_prefix(info, outs[b]);
        cuda_check(cudaMemcpyAsync(outs[b] + sbw::kDataOffset, d_in + b * words, words * sizeof(u64), cudaMemcpyDeviceToHost, st), "D2H");
    }
    cuda_check(cudaStreamSynchronize(st), "synchronize");
    return SB200_OK;
    SB_CATCH
}

// ---- decryption (SURVEY 8f rank 4): Decryptor(context, secret_key) + Decryptor::decrypt ----
int sb200_secret_key_create(sb200_context *ctx, const uint64_t *h_secret_key, sb200_secret_key **out)
{
    SB_NEED(h_secret_key);
    SB_NEED(out);
    SB_TRY
    SB_ENTER(ctx)
    auto h = std::make_unique<sb200_secret_key>();
    secret_key_create(c, (const u64 *)h_secret_key, h->k);
    *out = h.release();
    return SB200_OK;
    SB_CATCH
}

int sb200_secret_key_destroy(sb200_secret_key *key)
{
    SB_NEED(key);
    delete key;
    return SB200_OK;
}

// ---- Encryptor(context, public_key)::encrypt_zero (sb_prng.cu) ----
int sb200_public_key_create(sb200_context *ctx, const uint64_t *h_public_key, sb200_public_key **out)
{
    SB_NEED(h_public_key);
    SB_NEED(out);
    SB_TRY
    SB_ENTER(ctx)
    auto h = std::make_unique<sb200_public_key>();
    public_key_create(c, (const u64 *)h_public_key, h->k);
    *out = h.release();
    return SB200_OK;
    SB_CATCH
}

int sb200_public_key_destroy(sb200_public_key *key)
{
    SB_NEED(key);
    delete key;
    return SB200_OK;
}

namespace
{
    // fresh PRNG seeds from the OS entropy source, as UniformRandomGeneratorFactory::create does (randomgen.cpp:34-50); wiped on scope exit
    struct FreshSeeds
    {
        std::vector<u64> words;
        explicit FreshSeeds(size_t batch) : words(batch * 8)
        {
            std::random_device rd("/dev/urandom");
            for (auto &w : words)
                w = (static_cast<u64>(rd()) << 32) | static_cast<u64>(rd());
        }
        ~FreshSeeds()
        {
            volatile u64 *w = words.data(); // the seeds determine the noise: do not leave them on the heap
            for (size_t i = 0; i < words.size(); i++)
                w[i] = 0;
        }
    };
} // namespace

int sb200_encrypt_zero_asymmetric(sb200_context *ctx, sb200_public_key *key, size_t L, size_t batch, const uint64_t *h_seeds, uint64_t *d_out,
                                  void *stream)
{
    SB_NEED(key);
    SB_NEED(d_out);
    SB_TRY
    SB_ENTER_STREAM(ctx, stream)
    check_level(c, L, batch);
    std::unique_ptr<FreshSeeds> fresh;
    if (!h_seeds)
    {
        fresh = std::make_unique<FreshSeeds>(batch);
        h_seeds = reinterpret_cast<const uint64_t *>(fresh->words.data());
    }
    // returns after a stream synchronisation: the seeds may be wiped
    op_encrypt_zero_asymmetric(c, key->k, L, batch, (const u64 *)h_seeds, (u64 *)d_out, static_cast<cudaStream_t>(stream));
    return SB200_OK;
    SB_CATCH
}

// ---- CKKSEncoder::encode / decode (sb_ckks.cu) ----
int sb200_ckks_encode(sb200_context *ctx, size_t L, size_t batch, const double *d_values, size_t count, int is_complex, double scale,
                      uint64_t *d_plain, void *stream)
{
    SB_NEED(d_plain);
    SB_TRY
    SB_ENTER_STREAM(ctx, stream)
    check_level(c, L, batch);
    op_ckks_encode(c, L, batch, d_values, count, is_complex != 0, scale, (u64 *)d_plain, static_cast<cudaStream_t>(stream));
    return SB200_OK;
    SB_CATCH
}

int sb200_ckks_decode(sb200_context *ctx, size_t L, size_t batch, const uint64_t *d_plain, double scale, double *d_values, void *stream)
{
    SB_NEED(d_plain);
    SB_NEED(d_values);
    SB_TRY
    SB_ENTER_STREAM(ctx, stream)
    check_level(c, L, batch);
    op_ckks_decode(c, L, batch, (const u64 *)d_plain, scale, d_values, static_cast<cudaStream_t>(stream));
    return SB200_OK;
    SB_CATCH
}

namespace
{
    struct DevBuf // scoped device allocation of the (not hot) host-buffer encoder entry points
    {
        void *p = nullptr;
        explicit DevBuf(size_t bytes)
        {
            cuda_check(cudaMalloc(&p, bytes ? bytes : 16), "cudaMalloc");
        }
        ~DevBuf()
        {
            cudaFree(p);
        }
        DevBuf(const DevBuf &) = delete;
        DevBuf &operator=(const DevBuf &) = delete;
    };
} // namespace

int sb200_ckks_encode_host(sb200_context *ctx, size_t L, size_t batch, const double *h_values, size_t count, int is_complex, double scale,
                           uint64_t *h_plain)
{
    SB_NEED(h_plain);
    SB_TRY
    SB_ENTER_STREAM(ctx, nullptr)
    check_level(c, L, batch);
    if (count && !h_values)
        throw std::invalid_argument("values cannot be null");
    const size_t vbytes = batch * count * (is_complex ? 16 : 8), pbytes = batch * L * c.n * sizeof(u64);
    DevBuf v(vbytes), p(pbytes);
    if (vbytes)
        cuda_check(cudaMemcpy(v.p, h_values, vbytes, cudaMemcpyHostToDevice), "values H2D");
    op_ckks_encode(c, L, batch, static_cast<const double *>(v.p), count, is_complex != 0, scale, static_cast<u64 *>(p.p), nullptr);
    cuda_check(cudaMemcpy(h_plain, p.p, pbytes, cudaMemcpyDeviceToHost), "plain D2H");
    return SB200_OK;
    SB_CATCH
}

int sb200_ckks_decode_host(sb200_context *ctx, size_t L, size_t batch, const uint64_t *h_plain, double scale, double *h_values)
{
    SB_NEED(h_plain);
    SB_NEED(h_values);
    SB_TRY
    SB_ENTER_STREAM(ctx, nullptr)
    check_level(c, L, batch);
    const size_t vbytes = batch * (c.n / 2) * 16, pbytes = batch * L * c.n * sizeof(u64);
    DevBuf v(vbytes), p(pbytes);
    cuda_check(cudaMemcpy(p.p, h_plain, pbytes, cudaMemcpyHostToDevice), "plain H2D");
    op_ckks_decode(c, L, batch, static_cast<const u64 *>(p.p), scale, static_cast<double *>(v.p), nullptr);
    cuda_check(cudaMemcpy(h_values, v.p, vbytes, cudaMemcpyDeviceToHost), "values D2H");
    return SB200_OK;
    SB_CATCH
}

// Encryptor::encrypt_zero_symmetric for a batch (sb_prng.cu); h_bootstrap_seeds == nullptr: fresh seeds from the OS entropy source,
// as UniformRandomGeneratorFactory::create does through random_uint64 (randomgen.cpp:34-50)
int sb200_encrypt_zero_symmetric(sb200_context *ctx, sb200_secret_key *key, size_t L, size_t batch, const uint64_t *h_bootstrap_seeds,
                                 int save_seed, uint64_t *d_out, uint64_t *h_public_seeds, void *stream)
{
    SB_NEED(key);
    SB_NEED(d_out);
    SB_TRY
    SB_ENTER_STREAM(ctx, stream)
    check_level(c, L, batch);
    std::unique_ptr<FreshSeeds> fresh;
    if (!h_bootstrap_seeds)
    {
        fresh = std::make_unique<FreshSeeds>(batch);
        h_bootstrap_seeds = reinterpret_cast<const uint64_t *>(fresh->words.data());
    }
    op_encrypt_zero_symmetric(c, key->k, L, batch, (const u64 *)h_bootstrap_seeds, save_seed != 0, (u64 *)d_out, (u64 *)h_public_seeds,
                              static_cast<cudaStream_t>(stream));
    // op_encrypt_zero_symmetric synchronised the stream while expanding c_1: the seeds have been consumed and may be wiped
    return SB200_OK;
    SB_CATCH
}

} // extern "C"
