// Hand-written sm_100a kernels of the TAD engine.  See DESIGN.md for the pipeline:
//
//   hist     (K1)  columns -> key pack -> 64-bit hash -> bucket histogram      reads 17-21 B/row
//                  (exact path only: multi-GPU, or fallback of the optimistic partition)
//   bscan    (K1b) exclusive scan of the bucket counts, capacity-class lists, oversized-bucket list
//   scatter  (K2)  columns -> 32 B packed rows, hash-partitioned; on one GPU optimistically
//                  into fixed-capacity bucket slots with an overflow list      reads 29, writes 32 B/row
//   group    (K3)  one CTA per bucket: TMA bulk load into shared memory, hash-group by
//                  key, O(n) bucket-sort of each series by flowEndSeconds, reduce duplicates,
//                  write per-series arrays + series entries                   reads 32, writes 12 B/row
//   sscan    (K3b) exclusive scan of series-per-bucket
//   detect   (K4)  one thread per series straight out of csr_v: stddev_samp (Welford,
//                  sequential FP64), EWMA / DBSCAN score + flag, queued emission  reads 8-12 B/row
//
// All FP64 arithmetic on the score path uses explicit round-to-nearest intrinsics in the
// exact operation order of the reference UDFs (anomaly_detection.py:146-212) so that the
// results are bit-identical to the CPU oracle (no FMA contraction).
#include "tad_kernels.h"

#include <atomic>
#include <cstdio>
#include <mutex>

namespace tad {

// ----------------------------------------------------------------------------------------
// small PTX helpers
// ----------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 ldg_stream128(const void *p)
{
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ uint2 ldg_stream64(const void *p)
{
    uint2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
    return r;
}
// one 32-byte row = one 256-bit store = one full DRAM sector per request (sm_100: STG.E.256)
__device__ __forceinline__ void stg256(void *p, uint4 lo, uint4 hi)
{
    asm volatile("st.global.L1::no_allocate.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 :: "l"(p), "r"(lo.x), "r"(lo.y), "r"(lo.z), "r"(lo.w), "r"(hi.x), "r"(hi.y), "r"(hi.z), "r"(hi.w)
                 : "memory");
}
__device__ __forceinline__ uint32_t smem_u32(const void *p)
{
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ uint64_t pack64(uint32_t lo, uint32_t hi) { return ((uint64_t)hi << 32) | lo; }

// ----------------------------------------------------------------------------------------
// K1 / K2: histogram and scatter share the row loader
// ----------------------------------------------------------------------------------------
struct RowRegs {
    uint64_t a, b, value;
    uint32_t t, proto;
    bool keep;
};

__device__ __forceinline__ bool ns_ignored(const RowFilter &f, uint32_t ns)
{
    for (uint32_t i = 0; i < f.n_ns_ignore; i++)
        if (f.ns_ignore[i] == ns) return true;
    return false;
}

__device__ __forceinline__ bool row_keep(const RowFilter &f, const ColPtrs &c, uint64_t i, uint32_t fs, uint32_t fe)
{
    bool keep = true;
    if (f.start_time) keep = keep && (fs >= f.start_time);
    if (f.end_time) keep = keep && (fe < f.end_time);
    if (f.n_ns_ignore) {
        if (c.src_ns) keep = keep && !ns_ignored(f, c.src_ns[i]);
        if (c.dst_ns) keep = keep && !ns_ignored(f, c.dst_ns[i]);
    }
    return keep;
}

// Optimistic scatter (no histogram pass): every bucket owns a fixed slot of `cap` rows at part + bucket * cap;
// counters[] count arrivals from zero; a row whose arrival index is >= cap goes to the overflow list instead.
struct OptScatter {
    uint32_t cap;            // 0 = exact mode (counters hold absolute cursors)
    uint32_t ovf_cap;
    Row32 *ovf;
    uint32_t *ovf_count;
};

__device__ __forceinline__ void place_row(const RowRegs &r, uint32_t bucket, uint32_t pos, Row32 *part, const OptScatter &o)
{
    const uint4 lo = make_uint4((uint32_t)r.a, (uint32_t)(r.a >> 32), (uint32_t)r.b, (uint32_t)(r.b >> 32));
    const uint4 hi = make_uint4((uint32_t)r.value, (uint32_t)(r.value >> 32), r.t, r.proto);
    if (o.cap == 0) {
        stg256(part + pos, lo, hi);
    } else if (pos < o.cap) {
        stg256(part + (size_t)bucket * o.cap + pos, lo, hi);
    } else {
        const uint32_t k = atomicAdd(o.ovf_count, 1u);
        if (k < o.ovf_cap) stg256(o.ovf + k, lo, hi);
    }
}


// The scatter already has the 64-bit key hash in registers: the 24 bits right below the bucket bits travel with
// the row in the spare bytes of its protocol word, so the group kernel picks its hash slot without hashing again.
__device__ __forceinline__ uint32_t hash_tag(uint64_t h, int bshift)
{
    return (uint32_t)((h << (64 - min(bshift, 64))) >> 40);
}

template <bool SCATTER>
__device__ __forceinline__ void emit_row(const RowRegs &r, int bshift, uint32_t *counters, Row32 *part, const OptScatter &o)
{
    if (!r.keep) return;
    const uint64_t h = key_hash(r.a, r.b, r.proto);
    const uint32_t bucket = bshift >= 64 ? 0u : (uint32_t)(h >> bshift);
    if (SCATTER) {
        RowRegs rt = r;
        rt.proto |= hash_tag(h, bshift) << 8;
        place_row(rt, bucket, atomicAdd(&counters[bucket], 1u), part, o);
    } else {
        atomicAdd(&counters[bucket], 1u);
    }
}

__device__ __forceinline__ void load_row_scalar(const ColPtrs &c, const RowFilter &f, uint64_t i, bool need_tv, RowRegs &r)
{
    const uint32_t sip = c.src_ip ? c.src_ip[i] : 0u, dip = c.dst_ip ? c.dst_ip[i] : 0u;
    const uint32_t sp = c.src_port ? c.src_port[i] : 0u, dp = c.dst_port ? c.dst_port[i] : 0u;
    const uint32_t fs = c.flow_start ? c.flow_start[i] : 0u;
    const uint32_t fe = (need_tv || f.end_time) ? c.flow_end[i] : 0u;
    r.a = pack64(dip, sip);
    r.b = pack64((sp << 16) | dp, fs);
    r.proto = c.proto ? c.proto[i] : 0u;
    r.t = fe;
    r.value = need_tv ? c.value[i] : 0ull;
    r.keep = row_keep(f, c, i, fs, fe);
}

// 8 rows per thread, every column read with 128-bit (64-bit for the u8 column) streaming loads.
template <bool SCATTER, bool VEC>
__global__ void __launch_bounds__(256) partition_kernel(ColPtrs c, uint64_t R, RowFilter f, int bshift,
                                                        uint32_t *__restrict__ counters, Row32 *__restrict__ part,
                                                        const OptScatter opt)
{
    const uint64_t ngroups = (R + 7) / 8;
    const bool need_end = SCATTER || f.end_time != 0;
    for (uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; g < ngroups;
         g += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t base = g * 8;
        if (VEC && base + 8 <= R) {
            uint4 z = make_uint4(0, 0, 0, 0);
            uint4 sip0 = z, sip1 = z, dip0 = z, dip1 = z, fs0 = z, fs1 = z, fe0 = z, fe1 = z, sp = z, dp = z;
            uint4 v0 = z, v1 = z, v2 = z, v3 = z;
            uint2 pr = make_uint2(0, 0);
            if (c.src_ip) { sip0 = ldg_stream128(c.src_ip + base); sip1 = ldg_stream128(c.src_ip + base + 4); }
            if (c.dst_ip) { dip0 = ldg_stream128(c.dst_ip + base); dip1 = ldg_stream128(c.dst_ip + base + 4); }
            if (c.flow_start) { fs0 = ldg_stream128(c.flow_start + base); fs1 = ldg_stream128(c.flow_start + base + 4); }
            if (need_end) { fe0 = ldg_stream128(c.flow_end + base); fe1 = ldg_stream128(c.flow_end + base + 4); }
            if (c.src_port) sp = ldg_stream128(c.src_port + base);
            if (c.dst_port) dp = ldg_stream128(c.dst_port + base);
            if (c.proto) pr = ldg_stream64(c.proto + base);
            if (SCATTER) {
                v0 = ldg_stream128(c.value + base); v1 = ldg_stream128(c.value + base + 2);
                v2 = ldg_stream128(c.value + base + 4); v3 = ldg_stream128(c.value + base + 6);
            }
            const uint32_t sipv[8] = {sip0.x, sip0.y, sip0.z, sip0.w, sip1.x, sip1.y, sip1.z, sip1.w};
            const uint32_t dipv[8] = {dip0.x, dip0.y, dip0.z, dip0.w, dip1.x, dip1.y, dip1.z, dip1.w};
            const uint32_t fsv[8] = {fs0.x, fs0.y, fs0.z, fs0.w, fs1.x, fs1.y, fs1.z, fs1.w};
            const uint32_t fev[8] = {fe0.x, fe0.y, fe0.z, fe0.w, fe1.x, fe1.y, fe1.z, fe1.w};
            const uint32_t spw[4] = {sp.x, sp.y, sp.z, sp.w};
            const uint32_t dpw[4] = {dp.x, dp.y, dp.z, dp.w};
            const uint32_t vlo[8] = {v0.x, v0.z, v1.x, v1.z, v2.x, v2.z, v3.x, v3.z};
            const uint32_t vhi[8] = {v0.y, v0.w, v1.y, v1.w, v2.y, v2.w, v3.y, v3.w};
            RowRegs r[8];
#pragma unroll
            for (int i = 0; i < 8; i++) {
                const uint32_t sport = (spw[i >> 1] >> (16 * (i & 1))) & 0xffffu;
                const uint32_t dport = (dpw[i >> 1] >> (16 * (i & 1))) & 0xffffu;
                const uint32_t pw = i < 4 ? pr.x : pr.y;
                r[i].a = pack64(dipv[i], sipv[i]);
                r[i].b = pack64((sport << 16) | dport, fsv[i]);
                r[i].proto = (pw >> (8 * (i & 3))) & 0xffu;
                r[i].t = fev[i];
                r[i].value = pack64(vlo[i], vhi[i]);
                r[i].keep = row_keep(f, c, base + i, fsv[i], fev[i]);
            }
            if (SCATTER) {
                // all eight cursor atomics in flight before the first dependent store
                uint32_t pos[8], bkt[8];
#pragma unroll
                for (int i = 0; i < 8; i++) {
                    const uint64_t h = key_hash(r[i].a, r[i].b, r[i].proto);
                    bkt[i] = bshift >= 64 ? 0u : (uint32_t)(h >> bshift);
                    r[i].proto |= hash_tag(h, bshift) << 8;
                    pos[i] = r[i].keep ? atomicAdd(&counters[bkt[i]], 1u) : 0xffffffffu;
                }
#pragma unroll
                for (int i = 0; i < 8; i++)
                    if (r[i].keep) place_row(r[i], bkt[i], pos[i], part, opt);
            } else {
#pragma unroll
                for (int i = 0; i < 8; i++) emit_row<SCATTER>(r[i], bshift, counters, part, opt);
            }
        } else {
            const uint64_t end = base + 8 < R ? base + 8 : R;
            for (uint64_t i = base; i < end; i++) {
                RowRegs r;
                load_row_scalar(c, f, i, SCATTER, r);
                emit_row<SCATTER>(r, bshift, counters, part, opt);
            }
        }
    }
}

// ----------------------------------------------------------------------------------------
// multi-CTA exclusive scans (bucket offsets; series base per bucket).  The grid never exceeds the
// SM count with one 1024-thread CTA each, so all CTAs are co-resident and a CTA may spin on the
// partial sums its lower-numbered peers publish (flags carry a per-launch epoch: no memset).
// ----------------------------------------------------------------------------------------
constexpr int kScanMaxCtas = 128;
struct ScanSync {                       // lives in global memory, zero-initialised once
    unsigned long long part[kScanMaxCtas][4];
    unsigned int flag[kScanMaxCtas];
};

__device__ __forceinline__ uint32_t block_exclusive_scan_1024(uint32_t v, uint32_t *total)
{
    __shared__ uint32_t warp_sums[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t o = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += o;
    }
    __syncthreads();                    // protects warp_sums across back-to-back calls
    if (lane == 31) warp_sums[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        uint32_t w = warp_sums[lane];
        uint32_t winc = w;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            uint32_t o = __shfl_up_sync(0xffffffffu, winc, d);
            if (lane >= d) winc += o;
        }
        warp_sums[lane] = winc - w;
        if (lane == 31) *total = winc;
    }
    __syncthreads();
    return warp_sums[warp] + inc - v;
}

// publish this CTA's totals, then sum the totals of all lower CTAs (and of all CTAs)
__device__ __forceinline__ void grid_prefix(ScanSync *sy, uint32_t epoch, const unsigned long long mine[4],
                                            unsigned long long before[4], unsigned long long all[4])
{
    __shared__ unsigned long long sh_before[4], sh_all[4];
    const uint32_t c = blockIdx.x, G = gridDim.x;
    if (threadIdx.x == 0) {
        for (int k = 0; k < 4; k++) sy->part[c][k] = mine[k];
        __threadfence();
        atomicExch(&sy->flag[c], epoch);
    }
    if (threadIdx.x < 32) {
        unsigned long long b[4] = {0, 0, 0, 0}, a[4] = {0, 0, 0, 0};
        for (uint32_t o = threadIdx.x; o < G; o += 32) {
            while (atomicAdd(&sy->flag[o], 0u) != epoch) { }
            __threadfence();
            for (int k = 0; k < 4; k++) {
                const unsigned long long x = *reinterpret_cast<volatile unsigned long long *>(&sy->part[o][k]);
                a[k] += x;
                if (o < c) b[k] += x;
            }
        }
        for (int k = 0; k < 4; k++) {
            for (int d = 16; d; d >>= 1) {
                b[k] += __shfl_xor_sync(0xffffffffu, b[k], d);
                a[k] += __shfl_xor_sync(0xffffffffu, a[k], d);
            }
        }
        if (threadIdx.x == 0)
            for (int k = 0; k < 4; k++) { sh_before[k] = b[k]; sh_all[k] = a[k]; }
    }
    __syncthreads();
    for (int k = 0; k < 4; k++) { before[k] = sh_before[k]; all[k] = sh_all[k]; }
}

// offsets[B+1] = exclusive scan of hist; cursor = copy of offsets; lists the buckets larger
// than `cap` in ascending bucket order together with the exclusive scan of their sizes
// (big_base[n_big+1]) -- the spill path relies on that order.
__global__ void __launch_bounds__(1024) bucket_scan_kernel(const uint32_t *__restrict__ hist, uint32_t *__restrict__ offsets,
                                                           uint32_t *__restrict__ cursor, uint32_t B, uint32_t cap,
                                                           uint32_t *__restrict__ big_list, uint32_t *__restrict__ big_base,
                                                           uint32_t *__restrict__ cls_list /* 3 x B, may be null */,
                                                           uint32_t *__restrict__ stats, ScanSync *sy, uint32_t epoch)
{
    __shared__ uint32_t total_s, nbig_s, bigrows_s, maxb_s;
    if (threadIdx.x == 0) maxb_s = 0;
    const uint32_t per = (B + gridDim.x * 1024 - 1) / (gridDim.x * 1024);
    const uint32_t first = (blockIdx.x * 1024 + threadIdx.x) * per;
    const uint32_t lo = min(B, first), hi = min(B, first + per);
    uint32_t sum = 0, nbig = 0, bigrows = 0, mx = 0;
    for (uint32_t i = lo; i < hi; i++) {
        const uint32_t h = hist[i];
        sum += h;
        mx = max(mx, h);
        if (h > cap) { nbig++; bigrows += h; }
    }
    const uint32_t pre = block_exclusive_scan_1024(sum, &total_s);
    const uint32_t pre_nbig = block_exclusive_scan_1024(nbig, &nbig_s);
    const uint32_t pre_rows = block_exclusive_scan_1024(bigrows, &bigrows_s);
    atomicMax(&maxb_s, mx);
    __syncthreads();
    const unsigned long long mine[4] = {total_s, nbig_s, bigrows_s, maxb_s};
    unsigned long long before[4], all[4];
    grid_prefix(sy, epoch, mine, before, all);
    uint32_t run = (uint32_t)before[0] + pre, k = (uint32_t)before[1] + pre_nbig, br = (uint32_t)before[2] + pre_rows;
    for (uint32_t i = lo; i < hi; i++) {
        const uint32_t h = hist[i];
        offsets[i] = run;
        cursor[i] = run;
        run += h;
        if (h > cap) {
            big_list[k] = i;
            big_base[k] = br;
            k++;
            br += h;
        }
        if (cls_list) {
            // bucket list of its shared-memory capacity class (order is irrelevant: one CTA per entry);
            // one atomic per (warp, class) instead of one per bucket
            const uint32_t c = (h == 0 || h > cap) ? 3u : (h <= (uint32_t)kGroupCapSmall ? 0u : (h <= (uint32_t)kGroupCapMid ? 1u : 2u));
            const unsigned peers = __match_any_sync(__activemask(), c);
            if (c < 3u) {
                const int lane = threadIdx.x & 31, leader = __ffs(peers) - 1;
                uint32_t base = 0;
                if (lane == leader) base = atomicAdd(&stats[ST_NCLS0 + c], (uint32_t)__popc(peers));
                base = __shfl_sync(peers, base, leader);
                cls_list[(size_t)c * B + base + __popc(peers & ((1u << lane) - 1u))] = i;
            }
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        offsets[B] = (uint32_t)all[0];
        big_base[all[1]] = (uint32_t)all[2];
        stats[ST_KEPT] = (uint32_t)all[0];
        stats[ST_NBIG] = (uint32_t)all[1];
        stats[ST_BIGROWS] = (uint32_t)all[2];
    }
    if (threadIdx.x == 0) atomicMax(&stats[ST_MAXBUCKET], maxb_s);
}

// sbase[B+1] = exclusive scan of series-per-bucket, followed by the bucket hint table; also totals points.
__global__ void __launch_bounds__(1024) series_scan_kernel(const uint32_t *__restrict__ nsb, const uint32_t *__restrict__ npb,
                                                           uint32_t *__restrict__ sbase, uint32_t B, uint32_t *__restrict__ stats,
                                                           ScanSync *sy, uint32_t epoch)
{
    __shared__ uint32_t total_s;
    __shared__ unsigned long long points_s;
    if (threadIdx.x == 0) points_s = 0;
    __syncthreads();
    const uint32_t per = (B + gridDim.x * 1024 - 1) / (gridDim.x * 1024);
    const uint32_t first = (blockIdx.x * 1024 + threadIdx.x) * per;
    const uint32_t lo = min(B, first), hi = min(B, first + per);
    uint32_t sum = 0;
    unsigned long long pts = 0;
    for (uint32_t i = lo; i < hi; i++) { sum += nsb[i]; pts += npb[i]; }
    const uint32_t pre = block_exclusive_scan_1024(sum, &total_s);
    if (pts) atomicAdd(&points_s, pts);
    __syncthreads();
    const unsigned long long mine[4] = {total_s, points_s, 0, 0};
    unsigned long long before[4], all[4];
    grid_prefix(sy, epoch, mine, before, all);
    uint32_t run = (uint32_t)before[0] + pre;
    uint32_t *hint = sbase + B + 1;                 // hint[j] = bucket of series 32 * j (tad_common.cuh)
    for (uint32_t i = lo; i < hi; i++) {
        const uint32_t ns = nsb[i];
        sbase[i] = run;
        for (uint32_t m = (run + kHintStride - 1) & ~(kHintStride - 1); m < run + ns; m += kHintStride) hint[m / kHintStride] = i;
        run += ns;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        sbase[B] = (uint32_t)all[0];
        stats[ST_SERIES] = (uint32_t)all[0];
        stats[ST_POINTS] = (uint32_t)all[1];
    }
}

// ----------------------------------------------------------------------------------------
// K3: per-bucket group + time sort in shared memory
// ----------------------------------------------------------------------------------------
template <int CAP, int NT>
struct GroupSmem {
    static constexpr int HT = 2 * CAP;
    alignas(128) unsigned char x[32 * CAP];   // rows (TMA destination); later ts | tout | vout
    uint32_t ht[HT];                          // claim: low16 = rep row + 1, high16 = count; later (count << 16) | series idx
    uint16_t soff[HT];                        // first point of the slot's series inside the bucket
    alignas(8) unsigned long long mbar;
    uint32_t warp_sums[32];
    uint32_t total;
};

template <int NT>
__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t *warp_sums, uint32_t *total)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int NW = NT / 32;
    uint32_t inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t o = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += o;
    }
    if (lane == 31) warp_sums[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        uint32_t w = lane < NW ? warp_sums[lane] : 0u;
        uint32_t winc = w;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            uint32_t o = __shfl_up_sync(0xffffffffu, winc, d);
            if (lane >= d) winc += o;
        }
        if (lane < NW) warp_sums[lane] = winc - w;
        if (lane == NW - 1) *total = winc;
    }
    __syncthreads();
    return warp_sums[warp] + inc - v;
}


// Number of elements of a[lo, hi) that are < lim.  `a` is a 16-byte aligned shared-memory array;
// the body reads four elements per LDS.128 (lanes of one series read the same address -> broadcast).
__device__ __forceinline__ uint32_t count_lt_u32(const uint32_t *a, uint32_t lo, uint32_t hi, uint32_t lim)
{
    uint32_t c = 0, i = lo;
    const uint32_t head_end = min(hi, (lo + 3u) & ~3u);
    for (; i < head_end; i++) c += a[i] < lim ? 1u : 0u;
    const uint32_t body_end = i + ((hi - i) & ~3u);
#pragma unroll 2
    for (; i < body_end; i += 4) {
        const uint4 q = *reinterpret_cast<const uint4 *>(a + i);
        c += q.x < lim ? 1u : 0u;
        c += q.y < lim ? 1u : 0u;
        c += q.z < lim ? 1u : 0u;
        c += q.w < lim ? 1u : 0u;
    }
    for (; i < hi; i++) c += a[i] < lim ? 1u : 0u;
    return c;
}
__device__ __forceinline__ uint32_t count_lt_u64(const unsigned long long *a, uint32_t lo, uint32_t hi, unsigned long long lim)
{
    uint32_t c = 0, i = lo;
    const uint32_t head_end = min(hi, (lo + 1u) & ~1u);
    for (; i < head_end; i++) c += a[i] < lim ? 1u : 0u;
    const uint32_t body_end = i + ((hi - i) & ~1u);
#pragma unroll 4
    for (; i < body_end; i += 2) {
        const ulonglong2 q = *reinterpret_cast<const ulonglong2 *>(a + i);
        c += q.x < lim ? 1u : 0u;
        c += q.y < lim ? 1u : 0u;
    }
    for (; i < hi; i++) c += a[i] < lim ? 1u : 0u;
    return c;
}

constexpr int kSlotHashBits = 13;      // hash-tag bits that pick the shared-memory slot (largest table: 2 * kGroupCap)

template <int CAP, int NT, bool VRANK>
__global__ void __launch_bounds__(NT) group_kernel(const SegDesc seg, SeriesEntry *__restrict__ entries,
                                                   const uint32_t *__restrict__ offsets, const uint32_t *__restrict__ bucket_list,
                                                   uint32_t lo_rows,
                                                   uint64_t *__restrict__ csr_v, uint32_t *__restrict__ csr_t,
                                                   uint32_t *__restrict__ csr_p, uint32_t *__restrict__ nsb,
                                                   uint32_t *__restrict__ npb, int reducer)
{
    using S = GroupSmem<CAP, NT>;
    constexpr int HT = S::HT;
    constexpr int RPT = CAP / NT;      // rows per thread
    constexpr int SPT = HT / NT;       // hash slots per thread
    extern __shared__ __align__(128) unsigned char smem_raw[];
    S &s = *reinterpret_cast<S *>(smem_raw);

    const uint32_t bkt = bucket_list ? bucket_list[blockIdx.x] : blockIdx.x;
    const uint32_t off_b = offsets[bkt];
    const uint32_t n = offsets[bkt + 1] - off_b;
    const int tid = threadIdx.x;
    if (n <= lo_rows || n > (uint32_t)CAP) return;   // another capacity class (or the spill path) owns it

    // ---- L: one TMA bulk copy of the whole bucket into shared memory -----------------
    const uint32_t bar = smem_u32(&s.mbar);
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(1));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid < 32) {
        // one bulk copy per source segment, issued by up to 32 lanes in parallel: every lane fetches the
        // offsets of its own segment (one round of loads instead of nseg dependent rounds), a warp scan gives
        // the destination of each piece inside the staged bucket
        const uint32_t bytes = n * 32u;
        if (tid == 0) asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory");
        __syncwarp();
        uint32_t so = 0, sc = 0;
        if (tid < seg.nseg) seg_span(seg, tid, bkt, n, so, sc);
        uint32_t inc = sc;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t o = __shfl_up_sync(0xffffffffu, inc, d);
            if (tid >= d) inc += o;
        }
        if (sc)
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         :: "r"(smem_u32(s.x) + (inc - sc) * 32u), "l"(seg.base[tid] + so), "r"(sc * 32u), "r"(bar) : "memory");
    }
#pragma unroll
    for (int i = 0; i < SPT; i++) s.ht[tid + i * NT] = 0u;
    __syncthreads();
    {
        uint32_t done = 0;
        while (!done) {
            asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                         : "=r"(done) : "r"(bar), "r"(0) : "memory");
        }
    }

    // ---- G: hash-group rows by key (open addressing, linear probing) -------------------
    const uint4 *x4 = reinterpret_cast<const uint4 *>(s.x);
    uint32_t myT[RPT], mySP[RPT];
    uint64_t myV[RPT];
#pragma unroll
    for (int j = 0; j < RPT; j++) {
        const uint32_t r = tid + j * NT;
        myT[j] = 0; myV[j] = 0; mySP[j] = 0;
        if (r < n) {
            const uint4 k = x4[2 * r], w = x4[2 * r + 1];
            const uint32_t proto = w.w;                 // protocol | hash tag << 8 (equal keys carry equal tags)
            myT[j] = w.z;
            myV[j] = pack64(w.x, w.y);
            uint32_t slot = (proto >> (32 - kSlotHashBits)) & (HT - 1);
            while (true) {
                uint32_t cur = *reinterpret_cast<volatile uint32_t *>(&s.ht[slot]);
                if ((cur & 0xffffu) == 0u) {
                    const uint32_t old = atomicCAS(&s.ht[slot], 0u, r + 1u);
                    if (old == 0u) break;
                    cur = old;
                }
                const uint32_t rep = (cur & 0xffffu) - 1u;
                const uint4 kk = x4[2 * rep];
                const uint32_t pp = x4[2 * rep + 1].w;
                if (kk.x == k.x && kk.y == k.y && kk.z == k.z && kk.w == k.w && pp == proto) break;
                slot = (slot + 1) & (HT - 1);
            }
            const uint32_t pos = atomicAdd(&s.ht[slot], 0x10000u) >> 16;
            mySP[j] = slot | (pos << 16);
        }
    }
    __syncthreads();

    // ---- S: scan slot counts -> series offsets and dense series indices -----------------
    {
        const uint32_t base = tid * SPT;
        uint32_t loc[SPT];
        uint32_t sum = 0;
#pragma unroll
        for (int i = 0; i < SPT; i++) {
            const uint32_t w = s.ht[base + i];
            loc[i] = sum;
            sum += (w >> 16) | ((w & 0xffffu) ? 0x10000u : 0u);     // low16: points, high16: series
        }
        const uint32_t pre = block_exclusive_scan<NT>(sum, s.warp_sums, &s.total);
        SeriesEntry *ent = entries + off_b;
#pragma unroll
        for (int i = 0; i < SPT; i++) {
            const uint32_t w = s.ht[base + i];
            if (w & 0xffffu) {
                const uint32_t ex = pre + loc[i];
                const uint32_t so = ex & 0xffffu, k = ex >> 16, cnt = w >> 16, rep = (w & 0xffffu) - 1u;
                const uint4 kk = x4[2 * rep];
                const uint32_t pp = x4[2 * rep + 1].w;
                s.soff[base + i] = (uint16_t)so;
                s.ht[base + i] = (cnt << 16) | k;
                // series entry, in place over the (already staged) bucket rows
                uint4 *e4 = reinterpret_cast<uint4 *>(ent + k);
                e4[0] = kk;
                e4[1] = make_uint4(pp & 0xffu, cnt, off_b + so, 0u);
            }
        }
    }
    __syncthreads();                       // rows in s.x are dead from here on
    const uint32_t ns = s.total >> 16;

    uint32_t *ts = reinterpret_cast<uint32_t *>(s.x);                  // times in bin order (scratch)
    uint32_t *tout = ts + CAP;                                          // times, final order
    unsigned long long *vout = reinterpret_cast<unsigned long long *>(s.x + 8 * CAP);
    uint16_t *pslot = reinterpret_cast<uint16_t *>(s.x + 16 * CAP);   // VRANK: slot of the series at each position
    uint16_t *pout = reinterpret_cast<uint16_t *>(s.x + 18 * CAP);    // VRANK: value rank -> time index
    uint32_t *binc = reinterpret_cast<uint32_t *>(s.x + 20 * CAP);    // per-bin counts -> exclusive offsets
    uint32_t *tmin = reinterpret_cast<uint32_t *>(s.x + 24 * CAP);    // per series index
    uint32_t *tmax = reinterpret_cast<uint32_t *>(s.x + 28 * CAP);

    // ---- R: time-sort every series with an O(n) bucket sort ----------------------------------
    // A series of cnt points gets cnt bins over [tmin, tmax] (bin = trunc((t - tmin) * cnt / range),
    // monotone in t), bins are laid out series after series, so ONE block scan of the bin counts
    // yields every bin's final offset; rows of one bin (1-2 on average) are ordered by counting.
    for (uint32_t i = tid; i < n; i += NT) { binc[i] = 0u; tmin[i] = 0xffffffffu; tmax[i] = 0u; }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < RPT; j++) {
        const uint32_t r = tid + j * NT;
        if (r < n) {
            const uint32_t k = s.ht[mySP[j] & 0xffffu] & 0xffffu;
            atomicMin(&tmin[k], myT[j]);
            atomicMax(&tmax[k], myT[j]);
        }
    }
    __syncthreads();
    uint32_t myB[RPT];
#pragma unroll
    for (int j = 0; j < RPT; j++) {
        const uint32_t r = tid + j * NT;
        myB[j] = 0;
        if (r < n) {
            const uint32_t slot = mySP[j] & 0xffffu;
            const uint32_t w = s.ht[slot], so = s.soff[slot];
            const uint32_t cnt = w >> 16, k = w & 0xffffu;
            const uint32_t lo = tmin[k], range = tmax[k] - lo;
            uint32_t bin = 0;
            if (range) {
                const float scale = __uint2float_rn(cnt) / __uint2float_rn(range);
                bin = min(cnt - 1u, __float2uint_rz(__uint2float_rn(myT[j] - lo) * scale));
            }
            const uint32_t ord = atomicAdd(&binc[so + bin], 1u);
            myB[j] = (so + bin) | (ord << 16);
        }
    }
    __syncthreads();
    {   // exclusive scan of binc[0, n) in place
        uint32_t loc[RPT], sum = 0;
#pragma unroll
        for (int i = 0; i < RPT; i++) {
            const uint32_t q = tid * RPT + i;
            loc[i] = sum;
            sum += q < n ? binc[q] : 0u;
        }
        const uint32_t pre = block_exclusive_scan<NT>(sum, s.warp_sums, &s.total);
#pragma unroll
        for (int i = 0; i < RPT; i++) {
            const uint32_t q = tid * RPT + i;
            if (q < n) binc[q] = pre + loc[i];
        }
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < RPT; j++) {
        const uint32_t r = tid + j * NT;
        if (r < n) ts[binc[myB[j] & 0xffffu] + (myB[j] >> 16)] = myT[j];
    }
    __syncthreads();
    uint32_t anydup = 0;
#pragma unroll
    for (int j = 0; j < RPT; j++) {
        const uint32_t r = tid + j * NT;
        if (r < n) {
            const uint32_t slot = mySP[j] & 0xffffu;
            const uint32_t bi = myB[j] & 0xffffu, ord = myB[j] >> 16;
            const uint32_t b0 = binc[bi], b1 = bi + 1 < n ? binc[bi + 1] : n;
            const uint32_t t = myT[j];
            uint32_t pos = b0;
            for (uint32_t q = b0; q < b1; q++) {
                const uint32_t tq = ts[q];
                pos += (tq < t || (tq == t && q - b0 < ord)) ? 1u : 0u;
            }
            tout[pos] = t;
            vout[pos] = myV[j];
            if (VRANK) pslot[pos] = (uint16_t)slot;
            mySP[j] = pos | ((pos > s.soff[slot] ? 1u : 0u) << 31);
        }
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < RPT; j++) {
        const uint32_t r = tid + j * NT;
        if (r < n && (mySP[j] >> 31)) {
            const uint32_t p = mySP[j] & 0x7fffffffu;
            anydup |= (tout[p - 1] == myT[j]) ? 1u : 0u;
        }
    }
    uint32_t points = n;
    if (__syncthreads_or((int)anydup)) {
        // ---- D: rare -- reduce duplicates of (key, flowEndSeconds), one thread per slot ----
        SeriesEntry *ent = entries + off_b;
        uint32_t removed = 0;
        for (int i = 0; i < SPT; i++) {
            const uint32_t sl = tid * SPT + i;
            const uint32_t w = s.ht[sl];
            const uint32_t cnt = w >> 16;
            if (cnt < 2) continue;
            const uint32_t so = s.soff[sl];
            uint32_t wr = 0;
            for (uint32_t q = 1; q < cnt; q++) {
                if (tout[so + q] == tout[so + wr]) {
                    const unsigned long long x = vout[so + wr], y = vout[so + q];
                    vout[so + wr] = reducer == 0 ? (x > y ? x : y) : (x + y);
                } else {
                    ++wr;
                    tout[so + wr] = tout[so + q];
                    vout[so + wr] = vout[so + q];
                }
            }
            if (wr + 1 != cnt) {
                removed += cnt - (wr + 1);
                ent[w & 0xffffu].n = wr + 1;
                s.ht[sl] = ((wr + 1) << 16) | (w & 0xffffu);
            }
        }
        __syncthreads();
        const uint32_t pre = block_exclusive_scan<NT>(removed, s.warp_sums, &s.total);
        (void)pre;
        points = n - s.total;
    }

    if (VRANK) {
        // ---- V: rank every point inside its series by (value, time index) for the DBSCAN sweep ----
        __syncthreads();
        for (uint32_t p = tid; p < n; p += NT) {
            const uint32_t slot = pslot[p];
            const uint32_t so = s.soff[slot], cnt = s.ht[slot] >> 16, me = p - so;
            if (me >= cnt) continue;                    // hole left by the duplicate reduce
            const unsigned long long v = vout[p];
            uint32_t rank = (v == ~0ull) ? me : count_lt_u64(vout, so, so + me, v + 1ull);
            rank += count_lt_u64(vout, so + me, so + cnt, v);
            pout[so + rank] = (uint16_t)me;
        }
        __syncthreads();
    }

    // ---- W: coalesced write of the per-series arrays ------------------------------------
    for (uint32_t p = tid; p < n; p += NT) {
        csr_t[off_b + p] = tout[p];
        csr_v[off_b + p] = vout[p];
        if (VRANK) csr_p[off_b + p] = pout[p];
    }
    if (tid == 0) { nsb[bkt] = ns; npb[bkt] = points; }
}

// ----------------------------------------------------------------------------------------
// K4: detect -- one thread per series
// ----------------------------------------------------------------------------------------
// Bucket of series `i` for every thread of a CTA whose threads hold consecutive series: one thread searches
// the bucket of the CTA's first series, a window of sbase[] starting there is staged in shared memory, and
// each thread finishes with a short search inside the window (global binary search only if it falls outside).
constexpr int kBucketWindow = 256;
__device__ __forceinline__ uint32_t find_bucket_cta(const uint32_t *__restrict__ sbase, const uint32_t *__restrict__ offsets, uint32_t B,
                                                    uint32_t i, uint32_t i_first, uint32_t *win /* kBucketWindow + 1 */,
                                                    uint32_t *woff /* kBucketWindow + 1 */, uint32_t *b0_s)
{
    if (threadIdx.x == 0) *b0_s = find_bucket(sbase, B, i_first);
    __syncthreads();
    const uint32_t b0 = *b0_s;
    for (uint32_t k = threadIdx.x; k <= (uint32_t)kBucketWindow; k += blockDim.x) {
        win[k] = b0 + k <= B ? sbase[b0 + k] : 0xffffffffu;
        woff[k] = b0 + k <= B ? offsets[b0 + k] : 0u;      // same round trip: the entry address needs both
    }
    __syncthreads();
    if (win[kBucketWindow] <= i) return find_bucket(sbase, B, i);      // beyond the window (many empty buckets)
    uint32_t lo = 0, hi = kBucketWindow;                                // win[lo] <= i < win[hi]
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (win[mid] <= i) lo = mid; else hi = mid;
    }
    return b0 + lo;
}

__device__ __forceinline__ void write_out(const OutCols &o, uint32_t idx, const SeriesEntry &e, uint32_t t, double sd,
                                          double calc, double x, bool flag)
{
    o.src_ip[idx] = (uint32_t)(e.a >> 32);
    o.dst_ip[idx] = (uint32_t)e.a;
    o.flow_start[idx] = (uint32_t)(e.b >> 32);
    o.src_port[idx] = (uint16_t)(e.b >> 16);
    o.dst_port[idx] = (uint16_t)e.b;
    o.proto[idx] = (uint8_t)e.proto;
    o.flow_end[idx] = t;
    o.stddev[idx] = sd;
    o.algo_calc[idx] = calc;
    o.throughput[idx] = x;
    o.anomaly[idx] = flag ? 1 : 0;
}

// Division by the running count on the Welford critical path.  d / k with k a small integer is computed as
// q0 = d * r (r = RN(1/k) from a table filled with __drcp_rn) plus ONE FMA residual correction
// q1 = fma(fma(-k, q0, d), r, q0).  That is the correctly rounded quotient: q0 is within 1.5 ulp of z = d/k, so the
// residual k (z - q0) is exact, and q0 + residual * r = z + (z - q0) * eps with |eps| <= 2^-53 -- a perturbation
// below 2^-52 ulp(z) -- while z itself keeps a distance of at least ulp(z) / (2k) from every rounding boundary
// (d - k * midpoint is a non-zero multiple of ulp(z)/2).  So RN(q0 + residual * r) = RN(z) for every k < 2^50.
// Checked against `/` on 6e8 random and 1.2e9 near-midpoint operands (profiles/microbench/divcheck.c); three
// dependent operations instead of the ~30 of the generic __ddiv_rn sequence.
constexpr uint32_t kRcpTable = 4096;
__device__ double g_rcp[kRcpTable + 1];

__global__ void rcp_table_kernel()
{
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k <= kRcpTable) g_rcp[k] = k ? __drcp_rn((double)k) : 0.0;
}

// stddev_samp as Spark's CentralMomentAgg computes it (Welford), sequential in time order.  The reciprocals
// of the next four counts are fetched before the dependent chain of the current four values starts, so the
// table load never sits on the critical path.
__device__ __forceinline__ double series_stddev(const uint64_t *__restrict__ v, uint32_t n, bool &has_sd)
{
    double cnt = 0.0, avg = 0.0, m2 = 0.0;
    auto step = [&](uint64_t raw, double r, bool have_r) {
        const double x = __ull2double_rn(raw);
        cnt = __dadd_rn(cnt, 1.0);
        const double d = __dsub_rn(x, avg);
        double dn;
        if (have_r) {
            const double q0 = __dmul_rn(d, r);
            dn = __fma_rn(__fma_rn(-cnt, q0, d), r, q0);
        } else {
            dn = __ddiv_rn(d, cnt);
        }
        avg = __dadd_rn(avg, dn);
        m2 = __dadd_rn(m2, __dmul_rn(d, __dsub_rn(d, dn)));
    };
    uint32_t i = 0;
    const uint32_t mis = (uint32_t)((reinterpret_cast<uintptr_t>(v) >> 3) & 3u);
    const uint32_t head = min(n, (4u - mis) & 3u);
    for (; i < head; i++) step(v[i], g_rcp[min(i + 1u, kRcpTable)], i + 1u <= kRcpTable);
    double r0 = 0, r1 = 0, r2 = 0, r3 = 0;
    if (i + 4 <= n) {
        r0 = g_rcp[min(i + 1u, kRcpTable)]; r1 = g_rcp[min(i + 2u, kRcpTable)];
        r2 = g_rcp[min(i + 3u, kRcpTable)]; r3 = g_rcp[min(i + 4u, kRcpTable)];
    }
    for (; i + 4 <= n; i += 4) {
        const ulonglong2 a = *reinterpret_cast<const ulonglong2 *>(v + i);
        const ulonglong2 b = *reinterpret_cast<const ulonglong2 *>(v + i + 2);
        const double c0 = r0, c1 = r1, c2 = r2, c3 = r3;
        const bool ok = i + 4u <= kRcpTable;
        // reciprocals of the NEXT group: independent of the chain below
        r0 = g_rcp[min(i + 5u, kRcpTable)]; r1 = g_rcp[min(i + 6u, kRcpTable)];
        r2 = g_rcp[min(i + 7u, kRcpTable)]; r3 = g_rcp[min(i + 8u, kRcpTable)];
        step(a.x, c0, ok); step(a.y, c1, ok); step(b.x, c2, ok); step(b.y, c3, ok);
    }
    for (; i < n; i++) step(v[i], g_rcp[min(i + 1u, kRcpTable)], i + 1u <= kRcpTable);
    has_sd = n >= 2;
    return has_sd ? __dsqrt_rn(__ddiv_rn(m2, __dsub_rn(cnt, 1.0))) : __longlong_as_double(0x7ff8000000000000LL);
}

// ----------------------------------------------------------------------------------------
// K4 (EWMA): no shared-memory stage.  A thread streams its own series straight out of csr_v, one full
// 32-byte sector (four values, ONE 256-bit load through the read-only path) per step with the next sector already
// in flight, so no sector is fetched twice and the kernel runs at register-limited occupancy (5 CTAs of 128 threads
// per SM instead of two of 96).  The round-1 detector staged each CTA's span in shared memory with TMA and was latency
// bound -- 6 warps per SM on dependent FP64 chains issue ~0.75 instructions per clock and SM
// (profiles/r01_source_lines_detect.txt) -- and this one attacks exactly that with more warps.  Sectors are addressed from the sector-aligned start of the series (csr_v is padded by one sector),
// elements outside [0, n) are masked.  Flagged points are queued in shared memory (one warp-aggregated atomic per
// flagged point) and written out cooperatively, every result column coalesced.
// ----------------------------------------------------------------------------------------
constexpr int kDirectThreads = 128;
constexpr int kDirectQueue = 2048;                    // queued result rows per CTA (16 per series; the bench table has ~9)

struct DirectSmem {
    double qcalc[kDirectQueue];
    uint32_t qpos[kDirectQueue];
    uint32_t qmeta[kDirectQueue];                     // bit 31: flag, bits 30..16: owning thread
    unsigned long long ent_a[kDirectThreads], ent_b[kDirectThreads];
    double ent_sd[kDirectThreads];
    uint32_t ent_proto[kDirectThreads];
    uint32_t qcount, base, b0;
    uint32_t win[kBucketWindow + 1], woff[kBucketWindow + 1];
};

struct Sector4 { unsigned long long v[4]; };
__device__ __forceinline__ Sector4 ldg_sector(const uint64_t *p)      // p is 32-byte aligned
{
    Sector4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u64 {%0,%1,%2,%3}, [%4];"
                 : "=l"(r.v[0]), "=l"(r.v[1]), "=l"(r.v[2]), "=l"(r.v[3]) : "l"(p));
    return r;
}
__device__ __forceinline__ uint32_t ldg_nc_u32(const uint32_t *p)
{
    uint32_t r;
    asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(r) : "l"(p));
    return r;
}
__device__ __forceinline__ unsigned long long ldg_nc_u64(const uint64_t *p)
{
    unsigned long long r;
    asm volatile("ld.global.nc.u64 %0, [%1];" : "=l"(r) : "l"(p));
    return r;
}

template <int NT>
__global__ void __launch_bounds__(NT, 5) detect_ewma_direct_kernel(const SeriesEntry *__restrict__ entries, const uint32_t *__restrict__ offsets,
                                                                   const uint32_t *__restrict__ sbase, uint32_t B, uint32_t S,
                                                                   const uint64_t *__restrict__ csr_v, const uint32_t *__restrict__ csr_t,
                                                                   OutCols out, uint32_t out_cap, uint32_t *__restrict__ stats, int emit_all)
{
    __shared__ DirectSmem sm;
    const uint32_t i = blockIdx.x * NT + threadIdx.x;
    if (threadIdx.x == 0) sm.qcount = 0u;
    SeriesEntry e;
    e.n = 0; e.off = 0; e.a = 0; e.b = 0; e.proto = 0;
    const uint32_t bkt = find_bucket_cta(sbase, offsets, B, i < S ? i : S - 1, blockIdx.x * NT, sm.win, sm.woff, &sm.b0);   // syncs
    if (i < S) {
        const uint32_t wk = bkt - sm.b0;
        const bool inwin = wk < (uint32_t)kBucketWindow;
        const uint32_t ob = inwin ? sm.woff[wk] : offsets[bkt], sb = inwin ? sm.win[wk] : sbase[bkt];
        const uint4 *p = reinterpret_cast<const uint4 *>(entries + ob + (i - sb));
        const uint4 k = p[0], w = p[1];
        e.a = pack64(k.x, k.y); e.b = pack64(k.z, k.w); e.proto = w.x; e.n = w.y; e.off = w.z;
    }
    const uint32_t n = e.n;
    const int mis = (int)(e.off & 3u);
    const uint64_t *vs = csr_v + (e.off & ~3u);                   // sector-aligned start of the series
    const uint32_t ng = n ? ((uint32_t)mis + n + 3u) >> 2 : 0u;   // sectors the series touches

    bool has_sd = false;
    double sd = 0.0;
    if (n) {
        // ---- pass 1: stddev_samp (Welford in time order; see series_stddev for the exact-division argument) ---------
        double cnt = 0.0, avg = 0.0, m2 = 0.0;
        Sector4 cur = ldg_sector(vs);
        // reciprocals of the counts, fetched ONE SECTOR AHEAD: the table load is then never on the Welford chain (in the first
        // capture of this kernel 25 % of the stall samples sat on q0 = d * rc[j] waiting for it, profiles/r02_source_lines_detect.txt)
        double rn[4];
#pragma unroll
        for (int j = 0; j < 4; j++) rn[j] = g_rcp[min((uint32_t)max(j + 1 - mis, 0), kRcpTable)];
        for (uint32_t g = 0; g < ng; g++) {
            Sector4 nxt = cur;
            if (g + 1 < ng) nxt = ldg_sector(vs + 4 * (g + 1));
            const int i0 = (int)(4 * g) - mis;                    // element index of the sector's first value
            const double rc[4] = {rn[0], rn[1], rn[2], rn[3]};
#pragma unroll
            for (int j = 0; j < 4; j++) rn[j] = g_rcp[min((uint32_t)max(i0 + 4 + j + 1, 0), kRcpTable)];
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const int idx = i0 + j;
                if (idx >= 0 && idx < (int)n) {
                    const double x = __ull2double_rn(cur.v[j]);
                    cnt = __dadd_rn(cnt, 1.0);
                    const double d = __dsub_rn(x, avg);
                    double dn;
                    if ((uint32_t)idx + 1u <= kRcpTable) {
                        const double q0 = __dmul_rn(d, rc[j]);
                        dn = __fma_rn(__fma_rn(-cnt, q0, d), rc[j], q0);
                    } else {
                        dn = __ddiv_rn(d, cnt);
                    }
                    avg = __dadd_rn(avg, dn);
                    m2 = __dadd_rn(m2, __dmul_rn(d, __dsub_rn(d, dn)));
                }
            }
            cur = nxt;
        }
        has_sd = n >= 2;
        sd = has_sd ? __dsqrt_rn(__ddiv_rn(m2, __dsub_rn(cnt, 1.0))) : __longlong_as_double(0x7ff8000000000000LL);
        sm.ent_a[threadIdx.x] = e.a; sm.ent_b[threadIdx.x] = e.b; sm.ent_proto[threadIdx.x] = e.proto;
        sm.ent_sd[threadIdx.x] = sd;
        // ---- pass 2: EWMA + flag; flagged points go to the CTA's queue ---------------------------------------------
        if (has_sd || emit_all) {
            double prev = 0.0;
            cur = ldg_sector(vs);
            for (uint32_t g = 0; g < ng; g++) {
                Sector4 nxt = cur;
                if (g + 1 < ng) nxt = ldg_sector(vs + 4 * (g + 1));
                const int i0 = (int)(4 * g) - mis;
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    const int idx = i0 + j;
                    if (idx >= 0 && idx < (int)n) {
                        const double x = __ull2double_rn(cur.v[j]);
                        prev = __dadd_rn(__dmul_rn(0.5, prev), __dmul_rn(0.5, x));
                        const bool flag = has_sd && (fabs(__dsub_rn(x, prev)) > sd);
                        if (flag || emit_all) {
                            const uint32_t slot = atomicAdd(&sm.qcount, 1u);
                            if (slot < (uint32_t)kDirectQueue) {
                                sm.qcalc[slot] = prev;
                                sm.qpos[slot] = e.off + (uint32_t)idx;
                                sm.qmeta[slot] = (flag ? 0x80000000u : 0u) | (threadIdx.x << 16);
                            } else {                                    // queue full: direct emission
                                const uint32_t o = atomicAdd(&stats[ST_OUTCOUNT], 1u);
                                if (o < out_cap) write_out(out, o, e, csr_t[e.off + (uint32_t)idx], sd, prev, x, flag);
                            }
                        }
                    }
                }
                cur = nxt;
            }
        }
    }
    __syncthreads();
    const uint32_t nq = min(sm.qcount, (uint32_t)kDirectQueue);
    if (threadIdx.x == 0) sm.base = nq ? atomicAdd(&stats[ST_OUTCOUNT], nq) : 0u;
    __syncthreads();
    // ---- cooperative emission: one result row per thread and step, every column written coalesced; flowEndSeconds and
    // throughput come through the read-only path, so the loads of a step are all in flight before its first store
    for (uint32_t j = threadIdx.x; j < nq; j += NT) {
        const uint32_t idx = sm.base + j;
        if (idx >= out_cap) continue;
        const uint32_t meta = sm.qmeta[j], pos = sm.qpos[j], owner = (meta >> 16) & 0x7fffu;
        const uint32_t t = ldg_nc_u32(csr_t + pos);
        const unsigned long long xv = ldg_nc_u64(csr_v + pos);
        const uint64_t ka = sm.ent_a[owner], kb = sm.ent_b[owner];
        out.src_ip[idx] = (uint32_t)(ka >> 32);
        out.dst_ip[idx] = (uint32_t)ka;
        out.flow_start[idx] = (uint32_t)(kb >> 32);
        out.src_port[idx] = (uint16_t)(kb >> 16);
        out.dst_port[idx] = (uint16_t)kb;
        out.proto[idx] = (uint8_t)sm.ent_proto[owner];
        out.flow_end[idx] = t;
        out.stddev[idx] = sm.ent_sd[owner];
        out.algo_calc[idx] = sm.qcalc[j];
        out.throughput[idx] = __ull2double_rn(xv);
        out.anomaly[idx] = (meta >> 31) ? 1 : 0;
    }
}

// ----------------------------------------------------------------------------------------
// K4 (DBSCAN): exact 1-D rule of sklearn's DBSCAN(min_samples=4, eps=2.5e8)
// (anomaly_detection.py:325-349; oracle/tad_oracle.py:calculate_dbscan_anomaly)
// ----------------------------------------------------------------------------------------
#define TAD_DBSCAN_EPS 250000000.0
#define TAD_DBSCAN_MIN 4u

// squared distance exactly as sklearn's brute-force radius search evaluates it (n <= 11)
__device__ __forceinline__ double sk_brute_d2(double xi, double xj)
{
    const double d = __dadd_rn(__dadd_rn(__dmul_rn(xi, xi), __dmul_rn(-2.0, __dmul_rn(xi, xj))), __dmul_rn(xj, xj));
    return d > 0.0 ? d : 0.0;
}
__device__ __forceinline__ bool within_eps(double a, double b) { return fabs(__dsub_rn(a, b)) <= TAD_DBSCAN_EPS; }

template <int NT>
__global__ void __launch_bounds__(NT) detect_dbscan_kernel(const SeriesEntry *__restrict__ entries, const uint32_t *__restrict__ offsets,
                                                           const uint32_t *__restrict__ sbase, uint32_t B, uint32_t S,
                                                           const uint64_t *__restrict__ csr_v, const uint32_t *__restrict__ csr_t,
                                                           uint32_t *__restrict__ csr_p, uint32_t *__restrict__ scratch_pc,
                                                           uint8_t *__restrict__ scratch_flag, OutCols out, uint32_t out_cap,
                                                           uint32_t *__restrict__ stats, int emit_all)
{
    __shared__ uint32_t warp_sums[32];
    __shared__ uint32_t total_s, base_s;
    const uint32_t i = blockIdx.x * NT + threadIdx.x;
    SeriesEntry e;
    e.n = 0;
    const uint64_t *v = nullptr;
    uint8_t *flag = nullptr;
    bool has_sd = false;
    double sd = 0.0;
    uint32_t count = 0;
    if (i < S) {
        const uint32_t b = find_bucket(sbase, B, i);
        const uint4 *p = reinterpret_cast<const uint4 *>(entries + offsets[b] + (i - sbase[b]));
        const uint4 k = p[0], w = p[1];
        e.a = pack64(k.x, k.y); e.b = pack64(k.z, k.w); e.proto = w.x; e.n = w.y; e.off = w.z; e.pad = w.w;
        v = csr_v + e.off;
        flag = scratch_flag + e.off;
        const uint32_t n = e.n;
        sd = series_stddev(v, n, has_sd);
        if (n <= 11) {
            const double r2 = TAD_DBSCAN_EPS * TAD_DBSCAN_EPS;
            uint32_t core = 0;
            for (uint32_t a = 0; a < n; a++) {
                const double xa = __ull2double_rn(v[a]);
                uint32_t c = 0;
                for (uint32_t q = 0; q < n; q++) c += (a == q || sk_brute_d2(xa, __ull2double_rn(v[q])) <= r2) ? 1u : 0u;
                core |= (c >= TAD_DBSCAN_MIN ? 1u : 0u) << a;
            }
            for (uint32_t a = 0; a < n; a++) {
                const double xa = __ull2double_rn(v[a]);
                bool reach = (core >> a) & 1u;
                for (uint32_t q = 0; q < n && !reach; q++)
                    reach = ((core >> q) & 1u) && (a == q || sk_brute_d2(xa, __ull2double_rn(v[q])) <= r2);
                flag[a] = reach ? 0 : 1;
                count += reach ? 0u : 1u;
            }
        } else {
            uint32_t *perm = csr_p + e.off;
            uint32_t *pc = scratch_pc + e.off;           // pc[k] = cores among sorted positions 0..k
            if (e.pad) {                                 // series from the spill path: rank by value here
                for (uint32_t a = 0; a < n; a++) {
                    const uint64_t va = v[a];
                    uint32_t rank = 0;
                    for (uint32_t q = 0; q < n; q++) {
                        const uint64_t vq = v[q];
                        rank += (vq < va || (vq == va && q < a)) ? 1u : 0u;
                    }
                    perm[rank] = a;
                }
            }
            uint32_t lo = 0, hi = 0, run = 0;
            for (uint32_t k = 0; k < n; k++) {
                const double xk = __ull2double_rn(v[perm[k]]);
                while (!within_eps(xk, __ull2double_rn(v[perm[lo]]))) lo++;
                if (hi < k) hi = k;
                while (hi + 1 < n && within_eps(__ull2double_rn(v[perm[hi + 1]]), xk)) hi++;
                run += (hi - lo + 1 >= TAD_DBSCAN_MIN) ? 1u : 0u;
                pc[k] = run;
            }
            lo = 0; hi = 0;
            for (uint32_t k = 0; k < n; k++) {
                const uint32_t pk = perm[k];
                const double xk = __ull2double_rn(v[pk]);
                while (!within_eps(xk, __ull2double_rn(v[perm[lo]]))) lo++;
                if (hi < k) hi = k;
                while (hi + 1 < n && within_eps(__ull2double_rn(v[perm[hi + 1]]), xk)) hi++;
                const uint32_t cores = pc[hi] - (lo ? pc[lo - 1] : 0u);
                flag[pk] = cores == 0 ? 1 : 0;
                count += cores == 0 ? 1u : 0u;
            }
        }
        if (emit_all) count = n;
    }
    const uint32_t pre = block_exclusive_scan<NT>(count, warp_sums, &total_s);
    if (threadIdx.x == 0) base_s = total_s ? atomicAdd(&stats[ST_OUTCOUNT], total_s) : 0u;
    __syncthreads();
    if (count == 0) return;
    uint32_t idx = base_s + pre;
    const uint32_t *t = csr_t + e.off;
    for (uint32_t q = 0; q < e.n; q++) {
        const bool f = flag[q] != 0;
        if (f || emit_all) {
            if (idx < out_cap) write_out(out, idx, e, t[q], sd, 0.0, __ull2double_rn(v[q]), f);
            idx++;
        }
    }
}

// ----------------------------------------------------------------------------------------
// launchers
// ----------------------------------------------------------------------------------------
// The launchers are called from one worker thread per context; several contexts may live in one process
// (bench.py keeps two jobs in flight), so the lazily initialised process-wide values below are atomics.
static std::atomic<int> g_num_sms{0};
static int num_sms()
{
    int n = g_num_sms.load(std::memory_order_relaxed);
    if (!n) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
        g_num_sms.store(n, std::memory_order_relaxed);
    }
    return n;
}

static bool cols_aligned16(const ColPtrs &c)
{
    auto ok = [](const void *p) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) & 15u) == 0; };
    return ok(c.src_ip) && ok(c.dst_ip) && ok(c.flow_start) && ok(c.flow_end) && ok(c.src_port) && ok(c.dst_port) &&
           ok(c.proto) && ok(c.value);
}

static uint32_t partition_grid(uint64_t R)
{
    const uint64_t groups = (R + 7) / 8;
    const uint64_t want = (groups + 255) / 256;
    const uint64_t cap = (uint64_t)num_sms() * 8;           // 8 resident CTAs of 256 threads per SM
    return (uint32_t)(want < cap ? (want ? want : 1) : cap);
}

cudaError_t launch_hist(cudaStream_t st, const ColPtrs &c, uint64_t R, const RowFilter &f, int logB, uint32_t *hist)
{
    if (R == 0) return cudaSuccess;
    const int bshift = 64 - logB;
    const OptScatter none{0, 0, nullptr, nullptr};
    if (cols_aligned16(c))
        partition_kernel<false, true><<<partition_grid(R), 256, 0, st>>>(c, R, f, bshift, hist, nullptr, none);
    else
        partition_kernel<false, false><<<partition_grid(R), 256, 0, st>>>(c, R, f, bshift, hist, nullptr, none);
    return cudaGetLastError();
}

cudaError_t launch_scatter(cudaStream_t st, const ColPtrs &c, uint64_t R, const RowFilter &f, int logB, uint32_t *cursor,
                           Row32 *part, uint32_t slot_cap, Row32 *ovf, uint32_t ovf_cap, uint32_t *ovf_count)
{
    if (R == 0) return cudaSuccess;
    const int bshift = 64 - logB;
    const OptScatter opt{slot_cap, ovf_cap, ovf, ovf_count};
    if (cols_aligned16(c))
        partition_kernel<true, true><<<partition_grid(R), 256, 0, st>>>(c, R, f, bshift, cursor, part, opt);
    else
        partition_kernel<true, false><<<partition_grid(R), 256, 0, st>>>(c, R, f, bshift, cursor, part, opt);
    return cudaGetLastError();
}

size_t scan_sync_bytes() { return sizeof(ScanSync); }

static uint32_t scan_grid(uint32_t B)
{
    uint32_t g = (B + 1023) / 1024;
    const uint32_t cap = (uint32_t)min(kScanMaxCtas, num_sms() - 4);     // all CTAs must be co-resident
    return g < 1 ? 1 : (g > cap ? cap : g);
}

cudaError_t launch_bucket_scan(cudaStream_t st, const uint32_t *hist, uint32_t *offsets, uint32_t *cursor, uint32_t B,
                               uint32_t cap, uint32_t *big_list, uint32_t *big_base, uint32_t *cls_list, uint32_t *stats,
                               void *scan_sync, uint32_t epoch)
{
    bucket_scan_kernel<<<scan_grid(B), 1024, 0, st>>>(hist, offsets, cursor, B, cap, big_list, big_base, cls_list, stats,
                                                     static_cast<ScanSync *>(scan_sync), epoch);
    return cudaGetLastError();
}

template <int CAP, int NT, bool VRANK>
static cudaError_t launch_group_class(cudaStream_t st, const SegDesc &seg, SeriesEntry *entries, const uint32_t *offsets,
                                      const uint32_t *bucket_list, uint32_t n_buckets, uint32_t lo_rows,
                                      uint64_t *csr_v, uint32_t *csr_t, uint32_t *csr_p, uint32_t *nsb, uint32_t *npb,
                                      int reducer)
{
    using S = GroupSmem<CAP, NT>;
    static std::atomic<bool> configured{false};
    auto kern = group_kernel<CAP, NT, VRANK>;
    if (!configured.load(std::memory_order_acquire)) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(S));
        if (e != cudaSuccess) return e;
        configured.store(true, std::memory_order_release);
    }
    if (n_buckets == 0) return cudaSuccess;
    kern<<<n_buckets, NT, sizeof(S), st>>>(seg, entries, offsets, bucket_list, lo_rows, csr_v, csr_t, csr_p, nsb, npb,
                                           reducer);
    return cudaGetLastError();
}

// Three shared-memory capacity classes (1024 / 2048 / 4096 rows): most buckets fit the first and run at the
// highest occupancy.  Each class is launched over ITS OWN bucket list (built by the bucket scan), one CTA per
// listed bucket -- launching all B CTAs per class and exiting early costs ~0.5 ms per class at 180 KB of shared
// memory per CTA.  Empty buckets keep the zeroes the caller memset into nsb / npb.
template <bool VRANK>
static cudaError_t launch_group_all(cudaStream_t st, const SegDesc &seg, SeriesEntry *entries, const uint32_t *offsets,
                                    uint32_t B, const uint32_t *cls_list, const uint32_t n_cls[3], uint64_t *csr_v,
                                    uint32_t *csr_t, uint32_t *csr_p, uint32_t *nsb, uint32_t *npb, int reducer, int *launches)
{
    *launches = 0;
    cudaError_t e = cudaSuccess;
    if (n_cls[2]) {
        e = launch_group_class<kGroupCap, 512, VRANK>(st, seg, entries, offsets, cls_list + 2 * (size_t)B, n_cls[2], kGroupCapMid,
                                                      csr_v, csr_t, csr_p, nsb, npb, reducer);
        ++*launches;
    }
    if (e == cudaSuccess && n_cls[1]) {
        e = launch_group_class<kGroupCapMid, 256, VRANK>(st, seg, entries, offsets, cls_list + B, n_cls[1], kGroupCapSmall,
                                                         csr_v, csr_t, csr_p, nsb, npb, reducer);
        ++*launches;
    }
    if (e == cudaSuccess) {
        e = launch_group_class<kGroupCapSmall, 256, VRANK>(st, seg, entries, offsets, cls_list, n_cls[0], 0, csr_v, csr_t,
                                                           csr_p, nsb, npb, reducer);
        *launches += n_cls[0] ? 1 : 0;
    }
    return e;
}

cudaError_t launch_group(cudaStream_t st, const SegDesc &seg, SeriesEntry *entries, const uint32_t *offsets, uint32_t B,
                         const uint32_t *cls_list, const uint32_t n_cls[3], uint64_t *csr_v, uint32_t *csr_t,
                         uint32_t *csr_p, uint32_t *nsb, uint32_t *npb, int reducer, int *launches)
{
    return csr_p ? launch_group_all<true>(st, seg, entries, offsets, B, cls_list, n_cls, csr_v, csr_t, csr_p, nsb, npb,
                                          reducer, launches)
                 : launch_group_all<false>(st, seg, entries, offsets, B, cls_list, n_cls, csr_v, csr_t, csr_p, nsb, npb,
                                           reducer, launches);
}

cudaError_t launch_series_scan(cudaStream_t st, const uint32_t *nsb, const uint32_t *npb, uint32_t *sbase, uint32_t B,
                               uint32_t *stats, void *scan_sync, uint32_t epoch)
{
    series_scan_kernel<<<scan_grid(B), 1024, 0, st>>>(nsb, npb, sbase, B, stats, static_cast<ScanSync *>(scan_sync), epoch);
    return cudaGetLastError();
}

static void ensure_rcp_table(cudaStream_t st)
{
    static std::once_flag once;       // a second context waits here until the table is complete
    std::call_once(once, [&] {
        rcp_table_kernel<<<(kRcpTable + 256) / 256, 256, 0, st>>>();
        cudaStreamSynchronize(st);      // once per process: other contexts (streams) of this device read the table too
    });
}

cudaError_t launch_detect_ewma(cudaStream_t st, const SeriesEntry *entries, const uint32_t *offsets, const uint32_t *sbase, uint32_t B,
                               uint32_t S, const uint64_t *csr_v, const uint32_t *csr_t, const OutCols &out,
                               uint32_t out_cap, uint32_t *stats, int emit_all)
{
    if (S == 0) return cudaSuccess;
    ensure_rcp_table(st);
    detect_ewma_direct_kernel<kDirectThreads><<<(S + kDirectThreads - 1) / kDirectThreads, kDirectThreads, 0, st>>>(
        entries, offsets, sbase, B, S, csr_v, csr_t, out, out_cap, stats, emit_all);
    return cudaGetLastError();
}

cudaError_t launch_detect_dbscan(cudaStream_t st, const SeriesEntry *entries, const uint32_t *offsets, const uint32_t *sbase,
                                 uint32_t B, uint32_t S, const uint64_t *csr_v, const uint32_t *csr_t, const uint32_t *csr_p,
                                 uint32_t *scratch_pc, uint8_t *scratch_flag, const OutCols &out, uint32_t out_cap,
                                 uint32_t *stats, int emit_all)
{
    if (S == 0) return cudaSuccess;
    constexpr int NT = 128;
    ensure_rcp_table(st);
    detect_dbscan_kernel<NT><<<(S + NT - 1) / NT, NT, 0, st>>>(entries, offsets, sbase, B, S, csr_v, csr_t,
                                                              const_cast<uint32_t *>(csr_p), scratch_pc, scratch_flag, out,
                                                              out_cap, stats, emit_all);
    return cudaGetLastError();
}

// ----------------------------------------------------------------------------------------
// multi-GPU: segment offsets of this rank's bucket range from the all-gathered histograms
// ----------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) segment_scan_kernel(const uint32_t *__restrict__ hist_all, uint32_t B_global, uint32_t b_lo,
                                                            uint32_t B_local, uint32_t *__restrict__ seg_off,
                                                            unsigned long long *__restrict__ seg_rows,
                                                            unsigned long long *__restrict__ seg_before /* may be null */)
{
    __shared__ uint32_t total_s;
    __shared__ unsigned long long before_s;
    const uint32_t r = blockIdx.x;
    if (seg_before) {
        // rows of source segment r that sit in front of this rank's bucket range inside r's (bucket-ordered) partition
        // buffer: where the peer-pull group kernel starts reading
        if (threadIdx.x == 0) before_s = 0ull;
        __syncthreads();
        const uint32_t *hb = hist_all + (size_t)r * B_global;
        unsigned long long acc = 0;
        for (uint32_t i = threadIdx.x; i < b_lo; i += 1024) acc += hb[i];
        for (int d = 16; d; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
        if ((threadIdx.x & 31) == 0 && acc) atomicAdd(&before_s, acc);
        __syncthreads();
        if (threadIdx.x == 0) seg_before[r] = before_s;
    }
    const uint32_t *h = hist_all + (size_t)r * B_global + b_lo;
    uint32_t *out = seg_off + (size_t)r * (B_local + 1);
    const uint32_t per = (B_local + 1023) / 1024;
    const uint32_t lo = min(B_local, threadIdx.x * per), hi = min(B_local, lo + per);
    uint32_t sum = 0;
    for (uint32_t i = lo; i < hi; i++) sum += h[i];
    const uint32_t pre = block_exclusive_scan_1024(sum, &total_s);
    uint32_t run = pre;
    for (uint32_t i = lo; i < hi; i++) { out[i] = run; run += h[i]; }
    if (threadIdx.x == 0) { out[B_local] = total_s; seg_rows[r] = total_s; }
}

__global__ void __launch_bounds__(256) segment_total_kernel(const uint32_t *__restrict__ hist_all, uint32_t B_global, uint32_t b_lo,
                                                            uint32_t B_local, int nseg, uint32_t *__restrict__ total)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < B_local; i += gridDim.x * blockDim.x) {
        uint32_t t = 0;
        for (int r = 0; r < nseg; r++) t += hist_all[(size_t)r * B_global + b_lo + i];
        total[i] = t;
    }
}

// ----------------------------------------------------------------------------------------
// multi-GPU, optimistic partition + peer pull: the arrival counters of this rank's bucket range, read out of every
// source rank's (IPC-mapped) counter array over NVLink.  cnt[s * B_local + b] = rows source s holds for local bucket b
// (they sit in slot b_lo + b of s's partition buffer), total[b] = the bucket's size.
// ----------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t ld_sys_u32(const uint32_t *p)
{
    uint32_t v;
    asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

__global__ void __launch_bounds__(256) gather_counts_kernel(const PeerCounters pc, int world, uint32_t b_lo, uint32_t B_local,
                                                            uint32_t slot, uint32_t *__restrict__ cnt, uint32_t *__restrict__ total)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < B_local; i += gridDim.x * blockDim.x) {
        uint32_t c[8], t = 0;
#pragma unroll
        for (int r = 0; r < 8; r++) c[r] = r < world ? ld_sys_u32(pc.p[r] + b_lo + i) : 0u;      // all loads in flight
#pragma unroll
        for (int r = 0; r < 8; r++) {
            if (r < world) {
                const uint32_t k = min(c[r], slot);
                cnt[(size_t)r * B_local + i] = k;
                t += k;
            }
        }
        total[i] = t;
    }
}

__global__ void __launch_bounds__(256) sum_counters_kernel(const uint32_t *__restrict__ a, uint32_t n, uint32_t *__restrict__ out)
{
    unsigned long long acc = 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) acc += a[i];
    for (int d = 16; d; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
    if ((threadIdx.x & 31) == 0 && acc) atomicAdd(out, (uint32_t)acc);
}

cudaError_t launch_gather_counts(cudaStream_t st, const PeerCounters &pc, int world, uint32_t b_lo, uint32_t B_local, uint32_t slot,
                                 uint32_t *cnt, uint32_t *total, const uint32_t *my_counters, uint32_t B_global, uint32_t *kept_out)
{
    if (world > 8) return cudaErrorInvalidValue;
    const uint32_t g1 = (B_local + 255) / 256, g2 = (B_global + 255) / 256;
    const uint32_t cap = (uint32_t)num_sms() * 8;
    gather_counts_kernel<<<g1 > cap ? cap : g1, 256, 0, st>>>(pc, world, b_lo, B_local, slot, cnt, total);
    sum_counters_kernel<<<g2 > cap ? cap : g2, 256, 0, st>>>(my_counters, B_global, kept_out);
    return cudaGetLastError();
}

cudaError_t launch_segment_scan(cudaStream_t st, const uint32_t *hist_all, uint32_t B_global, uint32_t b_lo, uint32_t B_local,
                                int nseg, uint32_t *seg_off, uint32_t *total, unsigned long long *seg_rows,
                                unsigned long long *seg_before)
{
    segment_scan_kernel<<<nseg, 1024, 0, st>>>(hist_all, B_global, b_lo, B_local, seg_off, seg_rows, seg_before);
    const uint32_t grid = (B_local + 255) / 256;
    segment_total_kernel<<<grid > 1184 ? 1184 : grid, 256, 0, st>>>(hist_all, B_global, b_lo, B_local, nseg, total);
    return cudaGetLastError();
}

}  // namespace tad
