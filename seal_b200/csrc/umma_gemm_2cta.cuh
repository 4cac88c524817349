// CTA-pair version of the 3xFP16 split GEMM (gemm_mode 5):  C[M,N] = A[M,K] * W[N,K]^T (+ bias, GELU, split).
//
// Why: the one-CTA kernel (umma_gemm.cuh) stages 96 KB of operands per k-block of 64 (A h1/h2 128 rows,
// W h1/h2 256 rows) for 12 MMAs = 1536 tensor cycles, i.e. 64 B/cycle/SM; times 148 SMs that is ~9.5 KB
// per cycle out of an L2 that delivers ~6.3 KB/cycle chip-wide (B300_MICROARCH.md "LTS throughput cap"),
// so the tensor pipe cannot be busy more than ~2/3 of the time -- which is what the profiles show
// (62-67 % on the large shapes).  Two CTAs of a cluster (one TPC) computing a 256x256 tile with
// tcgen05.mma.cta_group::2 each stage only their own 128 rows of A and HALF of the W tile
// (128 of its 256 rows): 64 KB per k-block per SM for the same 1536 cycles of MMAs (-33 % L2 traffic).
//
// Protocol (rank = %cluster_ctarank, leader = rank 0):
//   full[s]   leader's barrier only; count 1 (leader producer's arrive.expect_tx of BOTH CTAs' bytes); every
//             TMA of either CTA is a .cta_group::2 load completing on it.
//   empty[s]  one per CTA (count 1): the leader's MMA thread commits with .multicast::cluster to both.
//   tfull[b]  one per CTA (count 1): multicast commit when a K chunk's partial sums are complete.
//   tempty[b] leader's barrier only; count 2 x 16 epilogue warps; the peer's warps arrive remotely.
// Each CTA's TMEM holds the accumulator rows of its own 128 rows (two 256-column buffers).  Pair p walks
// pair-tiles p, p + #pairs, ...; a pair-tile = 256 rows x 256 columns.
//
// Output: the MMA warp can run only two chunks (half a K = 1024 tile) ahead of the epilogue, so every cycle an
// epilogue warp spends on a tile's output after its last chunk is a cycle the tensor pipe may wait.  Each
// epilogue warp therefore finishes 16 columns of its 32 x 64 block at a time into a 2 KB shared-memory slot laid
// out as a TMA box (lane = row) and hands the slot to one cp.async.bulk.tensor store; it waits for that store
// to have read the slot only before refilling it.  The tensor maps clip at M and N, so ragged edges need no
// code, and the raw partial sums of a K-sliced tail tile go out the same way through a map over `part`.
#pragma once
#include "umma_gemm.cuh"

namespace sealb200 {

constexpr int U2_STAGES = 3;
constexpr int U2_AB = UM * 128;                       // one A tile (h1 or h2): 128 rows x 128 B
constexpr int U2_WB = 128 * 128;                      // this CTA's half of the W tile: 128 rows x 128 B
constexpr int U2_STAGE = 2 * U2_AB + 2 * U2_WB;       // 64 KB
constexpr int U2_SLOT = 2048;                         // per epilogue warp: 32 rows x 16 fp32, or 32 x 16 h1 + 32 x 16 h2
constexpr int U2_SMEM = U2_STAGES * U2_STAGE + 1024 /*alignment*/ + UEPI_WARPS * U2_SLOT + 256 /*barriers*/;

__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the same smem offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t map_to_cta(uint32_t addr, uint32_t rank) {
    uint32_t r; asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank)); return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA load into THIS CTA's smem whose completion bytes are credited to a barrier that may live in the peer CTA
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, uint32_t bar_cluster_addr, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar_cluster_addr), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void umma_f16_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// arrives on the barrier at this smem offset in BOTH CTAs once the pair's MMAs issued so far have retired
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"((uint16_t)3) : "memory");
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
// shared -> global tensor store of one box at (c0 = column, c1 = row); elements outside the map are not written
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                 ::"l"(reinterpret_cast<uint64_t>(map)), "r"(src), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// generic-proxy writes to shared memory become visible to the bulk-copy (async) proxy
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ uint32_t pack_half2(__half lo, __half hi) {
    return (uint32_t)__half_as_ushort(lo) | ((uint32_t)__half_as_ushort(hi) << 16);
}

template <bool GELU>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(UTHREADS2, 1)
umma_gemm_f16x3_2cta_kernel(const __grid_constant__ CUtensorMap tmA_hi, const __grid_constant__ CUtensorMap tmA_lo,
                            const __grid_constant__ CUtensorMap tmW_hi, const __grid_constant__ CUtensorMap tmW_lo,
                            // output boxes of 16 columns x 32 rows: fp32 C (SWIZZLE_64B), or with split_out the fp16
                            // halves h1 / h2 (SWIZZLE_32B); tmPart = the fp32 K-slice partial sums of the tail tiles
                            const __grid_constant__ CUtensorMap tmOut, const __grid_constant__ CUtensorMap tmOut2,
                            const __grid_constant__ CUtensorMap tmPart,
                            int M, int N, int K, const float* __restrict__ bias, float w_unscale, int split_out, int n_fastest,
                            int* __restrict__ overflow, int full_items, int tail_s) {
    constexpr int BN = 256, KE = 64, NST = U2_STAGES;
    constexpr int kChunkBlocks = UKC16;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t slots = base + NST * U2_STAGE;               // 1024-aligned: the swizzle patterns repeat within a slot
    const uint32_t bars = slots + UEPI_WARPS * U2_SLOT;
    const uint32_t full0 = bars, empty0 = bars + 8 * NST;
    const uint32_t tfull0 = bars + 16 * NST, tempty0 = tfull0 + 16;
    const uint32_t slot = tempty0 + 16;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;

    const int m_tiles = (M + UM - 1) / UM, n_tiles = (N + BN - 1) / BN;
    const int pm_tiles = (m_tiles + 1) / 2;                     // pair-tiles along M (256 rows each)
    const int total = pm_tiles * n_tiles;
    const int num_k = K / KE;
    // Work list: items [0, full_items) are whole pair-tiles (all of K); the pair-tiles that would form a
    // mostly idle last wave are cut into tail_s K-slices each, so that wave costs 1/tail_s of a tile time:
    // item full_items + j = slice j % tail_s of pair-tile full_items + j / tail_s, raw partial sums stored to
    // rows [j * 256, j * 256 + 256) of tmPart (umma_tail_finish_kernel adds the slices in order).
    const int total_items = full_items + (total - full_items) * tail_s;
    struct Item { int tile, kb0, nkb, slot; };
    auto decode = [&](int item) {
        Item w;
        if (item < full_items) { w.tile = item; w.kb0 = 0; w.nkb = num_k; w.slot = -1; }
        else { const int j = item - full_items; w.tile = full_items + j / tail_s; w.nkb = num_k / tail_s; w.kb0 = (j % tail_s) * w.nkb; w.slot = j; }
        return w;
    };

    if (warp == 1 && lane == 0) {
        for (int s = 0; s < NST; ++s) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(tfull0 + 8 * b, 1); mbar_init(tempty0 + 8 * b, 2 * UEPI_WARPS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    } else if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                                         // the peer's barriers exist before anything targets them
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(slot));

    if (warp == 0) {
        if (lane == 0) {
            const uint32_t lead_full0 = map_to_cta(full0, 0);   // full barriers live in the leader CTA
            uint32_t it = 0;
            for (int item = pair; item < total_items; item += n_pairs) {
                const Item w = decode(item);
                const int pm = n_fastest ? w.tile / n_tiles : w.tile % pm_tiles, n_tile = n_fastest ? w.tile % n_tiles : w.tile / pm_tiles;
                const int row_a = (2 * pm + (int)rank) * UM;                 // this CTA's 128 rows of A
                const int row_w = n_tile * BN + (int)rank * 128;             // this CTA's half of the W tile
                for (int kb = w.kb0; kb < w.kb0 + w.nkb; ++kb, ++it) {
                    const int s = it % NST;
                    const uint32_t ph = (it / NST) & 1;
                    mbar_wait(empty0 + 8 * s, ph ^ 1);
                    const uint32_t st = base + s * U2_STAGE;
                    if (rank == 0) mbar_expect_tx(full0 + 8 * s, 2 * U2_STAGE);
                    const uint32_t fb = lead_full0 + 8 * s;
                    tma_load_2d_pair(st, &tmA_hi, fb, kb * KE, row_a);
                    tma_load_2d_pair(st + U2_AB, &tmA_lo, fb, kb * KE, row_a);
                    tma_load_2d_pair(st + 2 * U2_AB, &tmW_hi, fb, kb * KE, row_w);
                    tma_load_2d_pair(st + 2 * U2_AB + U2_WB, &tmW_lo, fb, kb * KE, row_w);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0 && rank == 0) {
            // D=F32 (1<<4), A=B=F16, K-major both, N>>3 at bit 17, M>>4 at bit 24 with M = 256 for the pair
            const uint32_t idesc = (1u << 4) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
            uint32_t it = 0, ch = 0;
            for (int item = pair; item < total_items; item += n_pairs) {
                const int num_k_item = decode(item).nkb;
                const int num_chunks = (num_k_item + kChunkBlocks - 1) / kChunkBlocks;
                int kb = 0;
                for (int c = 0; c < num_chunks; ++c, ++ch) {
                    const int buf = ch & 1;
                    mbar_wait(tempty0 + 8 * buf, ((ch >> 1) & 1) ^ 1);       // both CTAs' epilogues drained this buffer
                    tc_fence_after();
                    const uint32_t tacc = tmem_base + (uint32_t)(buf * BN);
                    const int kend = (kb + kChunkBlocks < num_k_item) ? kb + kChunkBlocks : num_k_item;
                    for (int k0 = kb; kb < kend; ++kb, ++it) {
                        const int s = it % NST;
                        const uint32_t ph = (it / NST) & 1;
                        mbar_wait(full0 + 8 * s, ph);
                        tc_fence_after();
                        const uint32_t st = base + s * U2_STAGE;
                        const uint64_t a_hi = umma_desc<128>(st), a_lo = umma_desc<128>(st + U2_AB);
                        const uint64_t w_hi = umma_desc<128>(st + 2 * U2_AB), w_lo = umma_desc<128>(st + 2 * U2_AB + U2_WB);
#pragma unroll
                        for (int k = 0; k < KE / 16; ++k) {
                            umma_f16_pair(tacc, a_lo + 2 * k, w_hi + 2 * k, idesc, (kb != k0) || (k != 0));
                            umma_f16_pair(tacc, a_hi + 2 * k, w_lo + 2 * k, idesc, 1);
                            umma_f16_pair(tacc, a_hi + 2 * k, w_hi + 2 * k, idesc, 1);
                        }
                        umma_commit_pair(empty0 + 8 * s);                    // both CTAs may refill this stage
                    }
                    umma_commit_pair(tfull0 + 8 * buf);                      // both CTAs' epilogues may drain the chunk
                }
            }
        }
    } else if (warp >= 4) {
        const int q = warp & 3;
        const int cg = (warp - 4) >> 2;
        const uint32_t lead_tempty0 = map_to_cta(tempty0, 0);
        const uint32_t stg = slots + (uint32_t)(warp - 4) * U2_SLOT;
        uint32_t ch = 0;
        for (int item = pair; item < total_items; item += n_pairs) {
            const int num_chunks = ((item < full_items ? num_k : num_k / tail_s) + kChunkBlocks - 1) / kChunkBlocks;
            float acc[64];
#pragma unroll
            for (int j = 0; j < 64; ++j) acc[j] = 0.f;
            for (int c = 0; c < num_chunks; ++c, ++ch) {
                const int buf = ch & 1;
                mbar_wait(tfull0 + 8 * buf, (ch >> 1) & 1);
                tc_fence_after();
#pragma unroll
                for (int h = 0; h < 4; ++h) {                     // 16 columns at a time: 64 accumulators + 16 fresh values fit 96 registers
                    uint32_t r[16];
                    tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * BN + cg * 64 + h * 16), r);
#pragma unroll
                    for (int j = 0; j < 16; ++j) acc[h * 16 + j] += __uint_as_float(r[j]);
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_cluster(lead_tempty0 + 8 * buf);
            }
            const Item w = decode(item);                      // (kept out of the chunk loop: register pressure)
            const int pm = n_fastest ? w.tile / n_tiles : w.tile % pm_tiles, n_tile = n_fastest ? w.tile % n_tiles : w.tile / pm_tiles;
            const bool raw = w.slot >= 0;                     // K-slice of a tail tile: unscaled partial sums
            // this warp's 32 x 64 block: rows [row0, row0 + 32), columns [col0, col0 + 64) of C, or of the tail slice
            // (the rank is read again here so that nothing derived from it stays live across the chunk loop)
            const int rk = (int)cluster_ctarank();
            const int row0 = raw ? w.slot * 256 + rk * 128 + q * 32 : (2 * pm + rk) * UM + q * 32;
            const int col0 = raw ? cg * 64 : n_tile * BN + cg * 64;
            if (!raw && (row0 >= M || col0 >= N)) continue;
            // bias of the 64 columns, two per lane; column j is broadcast from lane j % 32 when it is needed
            float b_lo = 0.f, b_hi = 0.f;
            if (bias && !raw) {
                if (col0 + lane < N) b_lo = bias[col0 + lane];
                if (col0 + 32 + lane < N) b_hi = bias[col0 + 32 + lane];
            }
            int ov = 0;
#pragma unroll
            for (int pass = 0; pass < 4; ++pass) {            // 16 columns = one box per pass
                const int col = col0 + pass * 16;
                if (!raw && col >= N) break;
                float* v = acc + pass * 16;                   // finished in place
                if (!raw) {
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        const float x = v[j] * w_unscale + __shfl_sync(0xffffffffu, pass < 2 ? b_lo : b_hi, (pass * 16 + j) & 31);
                        v[j] = GELU ? gelu_erf_u(x) : x;
                    }
                }
                if (lane == 0) bulk_wait_read_all();          // the previous box has left the slot
                __syncwarp();
                if (split_out && !raw) {
                    // h1 at stg, h2 at stg + 1024: 32 B rows; SWIZZLE_32B puts 16-byte chunk c of row r at c ^ ((r >> 2) & 1)
                    uint32_t p1[8], p2[8];
#pragma unroll
                    for (int j = 0; j < 16; j += 2) {
                        __half a1, a2, c1, c2;
                        split_half(v[j], a1, a2, &ov);
                        split_half(v[j + 1], c1, c2, &ov);
                        p1[j / 2] = pack_half2(a1, c1);
                        p2[j / 2] = pack_half2(a2, c2);
                    }
#pragma unroll
                    for (int c = 0; c < 2; ++c) {
                        const uint32_t off = (uint32_t)(lane * 32 + ((c ^ ((lane >> 2) & 1)) * 16));
                        st_shared_v4(stg + off, p1[4 * c], p1[4 * c + 1], p1[4 * c + 2], p1[4 * c + 3]);
                        st_shared_v4(stg + 1024 + off, p2[4 * c], p2[4 * c + 1], p2[4 * c + 2], p2[4 * c + 3]);
                    }
                } else {
                    // fp32: 64 B rows; SWIZZLE_64B puts 16-byte chunk c of row r at c ^ ((r >> 1) & 3)
#pragma unroll
                    for (int c = 0; c < 4; ++c)
                        st_shared_v4(stg + (uint32_t)(lane * 64 + ((c ^ ((lane >> 1) & 3)) * 16)), __float_as_uint(v[4 * c]),
                                     __float_as_uint(v[4 * c + 1]), __float_as_uint(v[4 * c + 2]), __float_as_uint(v[4 * c + 3]));
                }
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) {
                    if (raw) tma_store_2d(&tmPart, stg, col, row0);
                    else if (split_out) { tma_store_2d(&tmOut, stg, col, row0); tma_store_2d(&tmOut2, stg + 1024, col, row0); }
                    else tma_store_2d(&tmOut, stg, col, row0);
                    bulk_commit();
                }
            }
            if (__any_sync(0xffffffffu, ov) && lane == 0) atomicExch(overflow, 1);
        }
        if (lane == 0) bulk_wait_all();
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                                         // nobody leaves while the pair's MMAs / remote arrives are in flight
    if (warp == 2) {
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// Finishes the K-sliced tail tiles of umma_gemm_f16x3_2cta_kernel: out = act((sum_s part[t][s]) * w_unscale + bias),
// slices added in index order (deterministic).  One thread per 4 consecutive columns of a 256 x 256 pair-tile.
template <bool GELU>
__global__ void __launch_bounds__(256) umma_tail_finish_kernel(int M, int N, int ldc, int n_tiles, int pm_tiles, int n_fastest,
                                                               int full_items, int tail_s, const float* __restrict__ part,
                                                               const float* __restrict__ bias, float w_unscale, float* __restrict__ C,
                                                               __half* __restrict__ C_h1, __half* __restrict__ C_h2, int* __restrict__ overflow) {
    const int t = blockIdx.x >> 6;                                // tail tile; 64 blocks of 256 threads x float4 each
    const int e = ((blockIdx.x & 63) << 8) + threadIdx.x;
    const int lr = e >> 6, c4 = e & 63;
    const int tile = full_items + t;
    const int pm = n_fastest ? tile / n_tiles : tile % pm_tiles, n_tile = n_fastest ? tile % n_tiles : tile / pm_tiles;
    const int row = pm * 256 + lr, n = n_tile * 256 + c4 * 4;
    if (row >= M || n >= N) return;
    const float* p = part + ((int64_t)t * tail_s * 256 + lr) * 256 + c4 * 4;
    float4 a = *reinterpret_cast<const float4*>(p);
    for (int sl = 1; sl < tail_s; ++sl) {
        const float4 b = *reinterpret_cast<const float4*>(p + (int64_t)sl * 65536);
        a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    }
    const float v[4] = {a.x, a.y, a.z, a.w};
    const int64_t off = (int64_t)row * ldc + n;
    int ov = 0;
    for (int u = 0; u < 4; ++u) {
        if (n + u >= N) continue;
        float x = v[u] * w_unscale + (bias ? bias[n + u] : 0.f);
        if (GELU) x = gelu_erf_u(x);
        if (C) C[off + u] = x;
        if (C_h1) { __half h1, h2; split_half(x, h1, h2, &ov); C_h1[off + u] = h1; C_h2[off + u] = h2; }
    }
    if (ov) atomicExch(overflow, 1);
}

}  // namespace sealb200
