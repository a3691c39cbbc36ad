// fa_simt.h -- thin SIMT vocabulary used by every kernel body in this directory.
//
// Compiled by nvcc (sm_100a) every name below maps 1:1 onto a CUDA intrinsic.  Compiled by a
// plain host C++ compiler (tests/hostsim only -- NEVER part of the shipped library) the same names
// are backed by an OS-thread-per-CUDA-thread emulator so that the block-cooperative kernel bodies
// can be unit-tested in the GPU-less build container before GPU minutes are spent.  The emulator
// is test infrastructure: libflacarray_b200.so contains only the CUDA instantiation and there is
// no CPU fallback in the product.
#pragma once
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
// ------------------------------------------------------------------------------------------------
// CUDA instantiation
// ------------------------------------------------------------------------------------------------
#define FA_D __device__ __forceinline__
#define FA_DNOINL __device__ __noinline__
#define FA_HD __host__ __device__ inline
#define FA_SHARED_BASE(name) extern __shared__ __align__(16) unsigned char name[]
#define FA_RESTRICT __restrict__

namespace fa {
FA_D int tid() { return (int)threadIdx.x; }
FA_D int nthreads() { return (int)blockDim.x; }
FA_D uint32_t blockIdx_x() { return blockIdx.x; }
FA_D uint32_t gridDim_x() { return gridDim.x; }
FA_D int lane() { return (int)(threadIdx.x & 31); }
FA_D int warp() { return (int)(threadIdx.x >> 5); }
FA_D void sync() { __syncthreads(); }
FA_D void syncwarp() { __syncwarp(); }
FA_D uint32_t shfl(uint32_t v, int src) { return __shfl_sync(0xffffffffu, v, src); }
FA_D uint32_t shfl_xor(uint32_t v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }
FA_D uint32_t shfl_up(uint32_t v, int d) { return __shfl_up_sync(0xffffffffu, v, d); }
FA_D uint32_t shfl_down(uint32_t v, int d) { return __shfl_down_sync(0xffffffffu, v, d); }
FA_D unsigned long long shfl64(unsigned long long v, int src) { return __shfl_sync(0xffffffffu, v, src); }
FA_D unsigned long long shfl_up64(unsigned long long v, int d) { return __shfl_up_sync(0xffffffffu, v, d); }
FA_D unsigned long long shfl_xor64(unsigned long long v, int m) {
    const uint32_t lo = shfl_xor((uint32_t)v, m), hi = shfl_xor((uint32_t)(v >> 32), m);
    return ((unsigned long long)hi << 32) | lo;
}
FA_D uint32_t ballot(bool p) { return __ballot_sync(0xffffffffu, p); }
FA_D int clz32(uint32_t v) { return __clz((int)v); }
FA_D int clz64(uint64_t v) { return __clzll((long long)v); }
FA_D int ctz32(uint32_t v) { return __ffs((int)v) - 1; }
FA_D int popc32(uint32_t v) { return __popc(v); }
FA_D uint32_t bswap32(uint32_t v) { return __byte_perm(v, 0, 0x0123); }
FA_D uint32_t funnel_l(uint32_t lo, uint32_t hi, uint32_t s) { return __funnelshift_l(lo, hi, s); }
// upper word of (hi:lo) << min(s, 32)
FA_D uint32_t funnel_lc(uint32_t lo, uint32_t hi, uint32_t s) { return __funnelshift_lc(lo, hi, s); }
// lower word of (hi:lo) >> (s & 31)
FA_D uint32_t funnel_r(uint32_t lo, uint32_t hi, uint32_t s) { return __funnelshift_r(lo, hi, s); }
// 0 or -1 from bit 0 (one SGXT)
FA_D int32_t sext1(uint32_t v) { int32_t r; asm("bfe.s32 %0, %1, 0, 1;" : "=r"(r) : "r"(v)); return r; }
FA_D uint32_t funnel_rc(uint32_t lo, uint32_t hi, uint32_t s) { return __funnelshift_rc(lo, hi, s); }   // s >= 32 -> hi
FA_D void atom_or_shared(uint32_t* p, uint32_t v) { atomicOr(p, v); }
FA_D void atom_add_shared64(unsigned long long* p, unsigned long long v) { atomicAdd(p, v); }
FA_D void atom_or_shared_u32(uint32_t* p, uint32_t v) { atomicOr(p, v); }
FA_D uint32_t atom_add_global(uint32_t* p, uint32_t v) { return atomicAdd(p, v); }
FA_D void atom_or_global(int* p, int v) { atomicOr(p, v); }
FA_D long long atom_cas_global64(long long* p, long long cmp, long long v) {
    return (long long)atomicCAS((unsigned long long*)p, (unsigned long long)cmp, (unsigned long long)v);
}
FA_D int atom_cas_global32(int* p, int cmp, int v) { return atomicCAS(p, cmp, v); }
FA_D void st_release_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
FA_D unsigned long long ld_acquire_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
FA_D void st_relaxed_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
FA_D unsigned long long ld_relaxed_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
FA_D void spin_pause() { __nanosleep(20); }
// 16-byte asynchronous copy global -> shared (LDGSTS): no destination register, so no scoreboard stall
FA_D void cp_async16(void* smem_dst, const void* gsrc) {
    uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
}
FA_D void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
FA_D void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
// ---- TMA bulk copy global -> shared, completion on an mbarrier (SASS: UBLKCP / SYNCS) -------------------
FA_D uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
FA_D void mbar_init(unsigned long long* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
// orders this thread's earlier generic-proxy accesses of shared memory before its later async-proxy (TMA) writes
FA_D void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// one thread: arm the barrier with the byte count and start the copy (16-byte aligned addresses, bytes % 16 == 0)
FA_D void bulk_load(void* smem_dst, const void* gsrc, uint32_t bytes, unsigned long long* bar) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// every consumer: block until the phase with this parity has completed
FA_D void mbar_wait(unsigned long long* bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
                     : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    } while (!ok);
}
// one thread: ask the L2 for `bytes` (a multiple of 16) from a 16-byte aligned global address; no destination, no wait
FA_D void prefetch_l2_bulk(const void* gsrc, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(gsrc), "r"(bytes) : "memory");
}
FA_D uint32_t ldg32(const uint32_t* p) { return __ldg(p); }
struct U4 { uint32_t x, y, z, w; };
FA_D U4 ldg128(const void* p) {  // 16-byte aligned, read-only path
    uint4 v = __ldg((const uint4*)p);
    U4 r; r.x = v.x; r.y = v.y; r.z = v.z; r.w = v.w;
    return r;
}
FA_D void sts128(void* p, U4 v) { *(uint4*)p = make_uint4(v.x, v.y, v.z, v.w); }   // 16-byte aligned shared/global store
FA_D U4 lds128(const void* p) { uint4 v = *(const uint4*)p; U4 r; r.x = v.x; r.y = v.y; r.z = v.z; r.w = v.w; return r; }
// |a - b| + acc in one instruction (VABSDIFF)
FA_D uint32_t sad_acc(int32_t a, int32_t b, uint32_t acc) { return __sad(a, b, acc); }
// warp-wide integer reductions (REDUX / CREDUX)
FA_D uint32_t redux_add(uint32_t v) { return __reduce_add_sync(0xffffffffu, v); }
FA_D uint32_t redux_or(uint32_t v) { return __reduce_or_sync(0xffffffffu, v); }
FA_D uint32_t redux_xor(uint32_t v) { return __reduce_xor_sync(0xffffffffu, v); }
FA_D int32_t redux_min(int32_t v) { return __reduce_min_sync(0xffffffffu, v); }
FA_D int32_t redux_max(int32_t v) { return __reduce_max_sync(0xffffffffu, v); }
FA_D float flog2(float v) { return __log2f(v); }
FA_D void st_global_u8x2(uint8_t* p, uint32_t hi, uint32_t lo) { p[0] = (uint8_t)hi; p[1] = (uint8_t)lo; }
// float ops with the rounding and (non-)contraction spelled out
FA_D float fadd(float a, float b) { return __fadd_rn(a, b); }
FA_D float fsub(float a, float b) { return __fsub_rn(a, b); }
FA_D float fmul(float a, float b) { return __fmul_rn(a, b); }
// trunc(a + b) of the exact sum, for |a + b| < 2^31: the round-towards-zero add never crosses an integer
FA_D int32_t trunc_fadd(float a, float b) { return __float2int_rz(__fadd_rz(a, b)); }
FA_D float fdiv(float a, float b) { return __fdiv_rn(a, b); }
FA_D double dadd(double a, double b) { return __dadd_rn(a, b); }
FA_D double dsub(double a, double b) { return __dsub_rn(a, b); }
FA_D double dmul(double a, double b) { return __dmul_rn(a, b); }
FA_D double ddiv(double a, double b) { return __ddiv_rn(a, b); }
FA_D double dfma(double a, double b, double c) { return __fma_rn(a, b, c); }
}  // namespace fa

#else
// ------------------------------------------------------------------------------------------------
// Host emulation (tests/hostsim only)
// ------------------------------------------------------------------------------------------------
#include <atomic>
#include <barrier>
#include <cmath>
#include <memory>
#include <thread>
#include <vector>

#define FA_D inline
#define FA_DNOINL inline
#define FA_HD inline
#define FA_RESTRICT __restrict__

namespace fasim {
struct Block {
    int nthreads;
    uint32_t nblocks = 1;
    std::barrier<> bar;
    std::vector<std::unique_ptr<std::barrier<>>> wbar;
    std::vector<uint64_t> xchg;  // one slot per thread
    std::vector<unsigned char> smem;
    explicit Block(int n, size_t smem_bytes) : nthreads(n), bar(n), xchg((size_t)n), smem(smem_bytes + 16) {
        for (int w = 0; w < (n + 31) / 32; ++w) {
            int cnt = (w + 1) * 32 <= n ? 32 : n - w * 32;
            wbar.emplace_back(new std::barrier<>(cnt));
        }
    }
};
struct ThreadCtx {
    Block* blk = nullptr;
    int tid = 0;
    int bid = 0;
};
extern thread_local ThreadCtx tls;

// Run `body(block_index)` for every block sequentially; each block = nthreads OS threads.
template <class F>
void launch(int nblocks, int nthreads, size_t smem_bytes, F body) {
    for (int b = 0; b < nblocks; ++b) {
        Block blk(nthreads, smem_bytes);
        blk.nblocks = (uint32_t)nblocks;
        std::vector<std::thread> th;
        for (int t = 0; t < nthreads; ++t) {
            th.emplace_back([&, t] {
                tls.blk = &blk;
                tls.tid = t;
                tls.bid = b;
                body(b);
            });
        }
        for (auto& x : th) x.join();
    }
}
inline unsigned char* smem() {
    uintptr_t p = (uintptr_t)tls.blk->smem.data();
    return (unsigned char*)((p + 15) & ~(uintptr_t)15);
}
}  // namespace fasim

#define FA_SHARED_BASE(name) unsigned char* name = fasim::smem()

namespace fa {
inline int tid() { return fasim::tls.tid; }
inline int nthreads() { return fasim::tls.blk->nthreads; }
inline uint32_t blockIdx_x() { return (uint32_t)fasim::tls.bid; }
inline uint32_t gridDim_x() { return fasim::tls.blk->nblocks; }
inline int lane() { return fasim::tls.tid & 31; }
inline int warp() { return fasim::tls.tid >> 5; }
inline void sync() { fasim::tls.blk->bar.arrive_and_wait(); }
inline void syncwarp() { fasim::tls.blk->wbar[(size_t)warp()]->arrive_and_wait(); }
inline uint64_t xchg_(uint64_t v, int src_lane) {
    auto* b = fasim::tls.blk;
    int base = fasim::tls.tid & ~31;
    b->xchg[(size_t)fasim::tls.tid] = v;
    syncwarp();
    int s = base + (src_lane & 31);
    uint64_t r = s < b->nthreads ? b->xchg[(size_t)s] : v;
    syncwarp();
    return r;
}
inline uint32_t shfl(uint32_t v, int src) { return (uint32_t)xchg_(v, src); }
inline uint32_t shfl_xor(uint32_t v, int m) { return (uint32_t)xchg_(v, lane() ^ m); }
inline uint32_t shfl_up(uint32_t v, int d) { return lane() - d >= 0 ? (uint32_t)xchg_(v, lane() - d) : ((void)xchg_(v, lane()), v); }
inline uint32_t shfl_down(uint32_t v, int d) { return lane() + d < 32 ? (uint32_t)xchg_(v, lane() + d) : ((void)xchg_(v, lane()), v); }
inline unsigned long long shfl64(unsigned long long v, int src) { return xchg_(v, src); }
inline unsigned long long shfl_up64(unsigned long long v, int d) { return lane() - d >= 0 ? xchg_(v, lane() - d) : ((void)xchg_(v, lane()), v); }
inline unsigned long long shfl_xor64(unsigned long long v, int m) { return xchg_(v, lane() ^ m); }
inline uint32_t ballot(bool p) {
    uint32_t r = 0;
    auto* b = fasim::tls.blk;
    int base = fasim::tls.tid & ~31;
    b->xchg[(size_t)fasim::tls.tid] = p ? 1u : 0u;
    syncwarp();
    for (int l = 0; l < 32 && base + l < b->nthreads; ++l) r |= (uint32_t)b->xchg[(size_t)(base + l)] << l;
    syncwarp();
    return r;
}
inline int clz32(uint32_t v) { return v ? __builtin_clz(v) : 32; }
inline int clz64(uint64_t v) { return v ? __builtin_clzll(v) : 64; }
inline int ctz32(uint32_t v) { return v ? __builtin_ctz(v) : -1; }
inline int popc32(uint32_t v) { return __builtin_popcount(v); }
inline uint32_t bswap32(uint32_t v) { return __builtin_bswap32(v); }
inline uint32_t funnel_l(uint32_t lo, uint32_t hi, uint32_t s) {
    s &= 31;
    return s ? (hi << s) | (lo >> (32 - s)) : hi;
}
inline uint32_t funnel_lc(uint32_t lo, uint32_t hi, uint32_t s) {
    if (s >= 32) return lo;
    return s ? (hi << s) | (lo >> (32 - s)) : hi;
}
inline uint32_t funnel_r(uint32_t lo, uint32_t hi, uint32_t s) {
    s &= 31;
    return s ? (lo >> s) | (hi << (32 - s)) : lo;
}
inline int32_t sext1(uint32_t v) { return -(int32_t)(v & 1u); }
inline uint32_t funnel_rc(uint32_t lo, uint32_t hi, uint32_t s) {
    if (s >= 32) return hi;
    return s ? (lo >> s) | (hi << (32 - s)) : lo;
}
inline void atom_or_shared(uint32_t* p, uint32_t v) { __atomic_fetch_or(p, v, __ATOMIC_RELAXED); }
inline void atom_add_shared64(unsigned long long* p, unsigned long long v) { __atomic_fetch_add(p, v, __ATOMIC_RELAXED); }
inline uint32_t atom_add_global(uint32_t* p, uint32_t v) { return __atomic_fetch_add(p, v, __ATOMIC_SEQ_CST); }
inline void atom_or_global(int* p, int v) { __atomic_fetch_or(p, v, __ATOMIC_SEQ_CST); }
inline long long atom_cas_global64(long long* p, long long cmp, long long v) {
    __atomic_compare_exchange_n(p, &cmp, v, false, __ATOMIC_SEQ_CST, __ATOMIC_SEQ_CST);
    return cmp;
}
inline int atom_cas_global32(int* p, int cmp, int v) {
    __atomic_compare_exchange_n(p, &cmp, v, false, __ATOMIC_SEQ_CST, __ATOMIC_SEQ_CST);
    return cmp;
}
inline void st_release_u64(unsigned long long* p, unsigned long long v) { __atomic_store_n(p, v, __ATOMIC_RELEASE); }
inline unsigned long long ld_acquire_u64(const unsigned long long* p) { return __atomic_load_n(p, __ATOMIC_ACQUIRE); }
inline void st_relaxed_u64(unsigned long long* p, unsigned long long v) { __atomic_store_n(p, v, __ATOMIC_RELAXED); }
inline unsigned long long ld_relaxed_u64(const unsigned long long* p) { return __atomic_load_n(p, __ATOMIC_RELAXED); }
inline void spin_pause() { std::this_thread::yield(); }
inline void cp_async16(void* smem_dst, const void* gsrc) { memcpy(smem_dst, gsrc, 16); }
inline void cp_async_commit() {}
inline void cp_async_wait_all() {}
inline void mbar_init(unsigned long long* bar, uint32_t) { *bar = 0; }
inline void fence_proxy_async() {}
// emulated barrier word = number of completed phases; the phase with parity p has completed when the count's parity differs
inline void bulk_load(void* smem_dst, const void* gsrc, uint32_t bytes, unsigned long long* bar) {
    memcpy(smem_dst, gsrc, bytes);
    __atomic_fetch_add(bar, 1ull, __ATOMIC_RELEASE);
}
inline void mbar_wait(unsigned long long* bar, uint32_t parity) {
    while ((__atomic_load_n(bar, __ATOMIC_ACQUIRE) & 1ull) == (unsigned long long)parity) std::this_thread::yield();
}
inline void prefetch_l2_bulk(const void*, uint32_t) {}
inline uint32_t ldg32(const uint32_t* p) { return *p; }
struct U4 { uint32_t x, y, z, w; };
inline U4 ldg128(const void* p) { U4 r; memcpy(&r, p, 16); return r; }
inline void sts128(void* p, U4 v) { memcpy(p, &v, 16); }
inline U4 lds128(const void* p) { U4 r; memcpy(&r, p, 16); return r; }
inline uint32_t sad_acc(int32_t a, int32_t b, uint32_t acc) {
    int64_t d = (int64_t)a - (int64_t)b;
    return acc + (uint32_t)(d < 0 ? -d : d);
}
template <class F>
inline uint32_t redux_(uint32_t v, F f) {
    auto* b = fasim::tls.blk;
    int base = fasim::tls.tid & ~31;
    b->xchg[(size_t)fasim::tls.tid] = v;
    syncwarp();
    uint32_t r = (uint32_t)b->xchg[(size_t)base];
    for (int l = 1; l < 32 && base + l < b->nthreads; ++l) r = f(r, (uint32_t)b->xchg[(size_t)(base + l)]);
    syncwarp();
    return r;
}
inline uint32_t redux_add(uint32_t v) { return redux_(v, [](uint32_t a, uint32_t b) { return a + b; }); }
inline uint32_t redux_or(uint32_t v) { return redux_(v, [](uint32_t a, uint32_t b) { return a | b; }); }
inline uint32_t redux_xor(uint32_t v) { return redux_(v, [](uint32_t a, uint32_t b) { return a ^ b; }); }
inline int32_t redux_min(int32_t v) { return (int32_t)redux_((uint32_t)v, [](uint32_t a, uint32_t b) { return (int32_t)a < (int32_t)b ? a : b; }); }
inline int32_t redux_max(int32_t v) { return (int32_t)redux_((uint32_t)v, [](uint32_t a, uint32_t b) { return (int32_t)a > (int32_t)b ? a : b; }); }
inline float flog2(float v) { return log2f(v); }
inline void st_global_u8x2(uint8_t* p, uint32_t hi, uint32_t lo) { p[0] = (uint8_t)hi; p[1] = (uint8_t)lo; }
// host build is compiled with -ffp-contract=off so these are the IEEE single operations
inline float fadd(float a, float b) { return a + b; }
inline float fsub(float a, float b) { return a - b; }
inline float fmul(float a, float b) { return a * b; }
inline int32_t trunc_fadd(float a, float b) { return (int32_t)((double)a + (double)b); }
inline float fdiv(float a, float b) { return a / b; }
inline double dadd(double a, double b) { return a + b; }
inline double dsub(double a, double b) { return a - b; }
inline double dmul(double a, double b) { return a * b; }
inline double ddiv(double a, double b) { return a / b; }
inline double dfma(double a, double b, double c) { return std::fma(a, b, c); }
}  // namespace fa
#endif
