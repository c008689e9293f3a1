// k_simgemm  --  the self-similarity contraction S = A A^T on the 5th-generation tensor cores.
//                                                            repet.py:1223 (_selfsimilaritymatrix)
// A = An32[rows][KPAD]: the normalised magnitude frames, K-major, KPAD = 1056 = 33 x 32 floats,
// pre-rounded to TF32 (round-to-nearest) by k_normalize.  Both operands are the same matrix.
//
// Warp-specialised, persistent (one CTA per SM, static tile schedule), sm_100a only:
//   warp 0      TMA producer: cp.async.bulk.tensor 128B-swizzled boxes [128 | 256 rows][32 floats]
//               into a 4-stage shared-memory ring, mbarrier expect_tx / complete_tx
//   warp 1      allocates TMEM (512 columns = two 128 x 256 fp32 accumulators) and issues
//               tcgen05.mma.cta_group::1.kind::tf32 (M 128, N 256, K 8) from one thread; smem stages
//               are released and accumulators published with tcgen05.commit
//   warps 2..5  epilogue: tcgen05.ld 32x32b.x32 (TMEM -> registers), transpose through a padded
//               smem tile so that global stores are 128-byte coalesced rows, predicated on the
//               ragged edges; overlaps the next tile's MMAs through the second accumulator
// In the split configuration only the tiles that reach the diagonal or lie above it are computed; the epilogue
// writes every element above the diagonal and its mirror image.  A row panel (tracks whose S exceeds the workspace
// limit) is computed as a full rectangle in both configurations.
// The result only PROPOSES similar-frame candidates: k_topk certifies every decision with exact
// float64 dot products, with tau covering the TF32 rounding (|S~ - S| <= 2 * 2^-11 + accumulation).
#include "repet_kernels.cuh"

#include <cuda.h>
#include <algorithm>
#include <cstdint>
#include <cstdio>

namespace repet {

namespace {

constexpr int BM = 128, BK = 32;  // BK floats = 128 bytes = one swizzle atom
constexpr int KBLOCKS = KPAD / BK;  // 33
constexpr int A_BYTES = BM * BK * 4;  // 16 KB
constexpr int EPI_PITCH = 33;
constexpr int EPI_BYTES = 4 * 32 * EPI_PITCH * 4;
constexpr int GEMM_THREADS = 192;

// Two configurations:
//   single pass  BN 256, 4 stages of (A 16 KB + B 32 KB): S~ = hi hi^T, |error| <= ~1e-3
//   split pass   BN 128, 3 stages of (A_hi, A_lo, B_hi, B_lo: 4 x 16 KB): A = hi + lo with both parts
//                TF32, S~ = hi hi^T + hi lo^T + lo hi^T accumulated in the same TMEM tile ("3xTF32",
//                fp32-class accuracy for 3x the MMAs)
template <int BN, bool SPLIT3>
struct GemmCfg {
    static constexpr int STAGES = SPLIT3 ? (BN == 256 ? 2 : 3) : 4;
    static constexpr int B_BYTES = BN * BK * 4;
    static constexpr int STAGE_BYTES = (SPLIT3 ? 2 : 1) * (A_BYTES + B_BYTES);
    static constexpr size_t SMEM = 1024 /*align slack*/ + (size_t)STAGES * STAGE_BYTES + EPI_BYTES + 256 /*barriers*/;
    static constexpr uint32_t TMEM_COLS = 2 * BN;  // two accumulators (power of two: 256 or 512)
    // instruction descriptor (cute::UMMA::InstrDescriptor): c=F32 [4,6), a=b=TF32 [7,10) [10,13), K-major
    // both, n_dim = N>>3 at [17,23), m_dim = M>>4 at [24,29)
    static constexpr uint32_t IDESC =
        (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// bounded wait: a protocol bug traps instead of hanging the GPU
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    for (uint32_t spin = 0; spin < (1u << 22); ++spin) {
        uint32_t done;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(addr), "r"(parity)
            : "memory");
        if (done) return;
    }
    printf("k_simgemm: mbarrier wait timed out (block %d thread %d)\n", (int)blockIdx.x, (int)threadIdx.x);
    __trap();
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
            smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(smem_u32(bar))
        : "memory");
}
// K-major, 128-byte swizzle: 8-row atoms 1024 bytes apart (SBO), version 1, layout type 2
__device__ __forceinline__ uint64_t umma_desc(const void* tile) {
    return (uint64_t)((smem_u32(tile) & 0x3ffffu) >> 4) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) |
           ((uint64_t)2 << 61);
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// Tile schedule.  S = A A^T is symmetric: with square tiles (the split configuration) only the tiles on and
// above the diagonal are computed and the epilogue writes each off-diagonal tile twice (once mirrored), which
// halves the MMAs.
// L2-aware raster: the operands of a 10-minute track (2 x 109 MB of hi / lo rows) do not fit the 126 MB L2, and a
// row-by-row walk of the triangle re-read every B block once per tile row (ncu, profiles/r2a_sim: 13.2 GB of DRAM
// reads for 218 MB of operands, L2 hit rate 61 %).  The triangle is cut into BANDS of RASTER_G tile rows; inside a
// band the tile COLUMN is the slow index and the row the fast one, so the 148 tiles in flight share the band's
// RASTER_G A blocks and ~10 B blocks (~28 MB) and every operand block comes from DRAM once per band.
constexpr int RASTER_G = 16;

// Triangle of tiles BM rows x BN columns, Q = BN / BM (1 or 2): tile (mi, nj) is computed iff it holds an element
// on or above the diagonal, i.e. nj >= mi / Q.  Band b holds tile rows [G b, G b + rb) and tile columns from
// c0 = (G / Q) b; its column c0 + c crosses rows r <= Q c + Q - 1, i.e. min(rb, Q (c + 1)) tiles.
template <int Q>
__host__ __device__ inline int band_tiles(int mt, int nt, int band, int* rb_out) {
    const int rb = min(RASTER_G, mt - RASTER_G * band);
    if (rb_out) *rb_out = rb;
    if (rb <= 0) return 0;
    const int nb = nt - (RASTER_G / Q) * band;
    int count = 0;
    for (int c = 0; c < nb; ++c) {
        const int h = min(rb, Q * (c + 1));
        if (h == rb) {
            count += (nb - c) * rb;
            break;
        }
        count += h;
    }
    return count;
}
template <int Q>
__host__ __device__ inline int triangle_tiles(int mt, int nt) {
    int total = 0;
    for (int band = 0; RASTER_G * band < mt; ++band) total += band_tiles<Q>(mt, nt, band, nullptr);
    return total;
}

// Without the triangle: row-major over the whole matrix, or (a row panel, `col_raster`) column by column -- all tile
// rows of a tile column before the next, so the panel's own operand rows stay in L2 while every other operand block
// is read once per panel (the band argument above with the panel as the band).
template <bool TRI, int Q>
__device__ __forceinline__ void decode_tile(int tile, int per_item, int mt, int nt, bool col_raster, int& item, int& mi,
                                            int& ni) {
    if (!TRI) {
        item = tile / (mt * nt);
        const int rem = tile - item * (mt * nt);
        if (col_raster) {
            ni = rem / mt;
            mi = rem - ni * mt;
        } else {
            mi = rem / nt;
            ni = rem - mi * nt;
        }
        return;
    }
    item = tile / per_item;
    int u = tile - item * per_item;
    int band = 0, rb = 0;
    for (;; ++band) {
        const int count = band_tiles<Q>(mt, nt, band, &rb);
        if (u < count || rb <= 0) break;
        u -= count;
    }
    int c = 0;
    for (;; ++c) {  // the columns that cross the diagonal (at most RASTER_G / Q of them), then full columns
        const int h = min(rb, Q * (c + 1));
        if (h == rb) {
            c += u / rb;
            u -= (u / rb) * rb;
            break;
        }
        if (u < h) break;
        u -= h;
    }
    mi = RASTER_G * band + u;
    ni = (RASTER_G / Q) * band + c;
}

// Rows [r0, r0 + rows) of S for every item: element (row, col) at S[(item * rows + row - r0) * T + col].  The whole
// matrix is r0 = 0, rows = T; TRI (the triangle with mirror writes) needs the whole matrix.
template <int BN, bool SPLIT3, bool TRI>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
k_simgemm(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
          const __grid_constant__ CUtensorMap map_a_lo, const __grid_constant__ CUtensorMap map_b_lo, int T, int r0,
          int rows, int n_items, int per_item, int col_raster, float* __restrict__ S) {
    using Cfg = GemmCfg<BN, SPLIT3>;
    constexpr int STAGES = Cfg::STAGES;
    constexpr int B_BYTES = Cfg::B_BYTES;
    constexpr int STAGE_BYTES = Cfg::STAGE_BYTES;
    constexpr uint32_t TMEM_COLS = Cfg::TMEM_COLS;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    unsigned char* tiles = smem;                                        // STAGES x (A | B), each 1024-aligned
    float* epi = reinterpret_cast<float*>(smem + STAGES * STAGE_BYTES);  // 4 x [32][33]
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES + EPI_BYTES);
    uint64_t* full = bars;                    // [STAGES]
    uint64_t* empty = bars + STAGES;          // [STAGES]
    uint64_t* acc_full = bars + 2 * STAGES;   // [2]
    uint64_t* acc_empty = acc_full + 2;       // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int Q = BN / BM;
    const int mt = (rows + BM - 1) / BM, nt = (T + BN - 1) / BN;
    const int row_end = r0 + rows;
    const int tiles_total = n_items * per_item;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&acc_full[a], 1);
            mbar_init(&acc_empty[a], 4);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "r"(TMEM_COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            uint32_t it = 0;
            for (int tile = blockIdx.x; tile < tiles_total; tile += gridDim.x) {
                int item, mi, ni;
                decode_tile<TRI, Q>(tile, per_item, mt, nt, col_raster, item, mi, ni);
                const int m0 = r0 + mi * BM, n0 = ni * BN;
                for (int kb = 0; kb < KBLOCKS; ++kb, ++it) {
                    const int s = it % STAGES;
                    mbar_wait(&empty[s], ((it / STAGES) & 1) ^ 1);
                    unsigned char* a_dst = tiles + (size_t)s * STAGE_BYTES;
                    mbar_arrive_expect_tx(&full[s], STAGE_BYTES);
                    tma_load_2d(a_dst, &map_a, kb * BK, item * T + m0, &full[s]);
                    tma_load_2d(a_dst + A_BYTES, &map_b, kb * BK, item * T + n0, &full[s]);
                    if (SPLIT3) {
                        tma_load_2d(a_dst + A_BYTES + B_BYTES, &map_a_lo, kb * BK, item * T + m0, &full[s]);
                        tma_load_2d(a_dst + 2 * A_BYTES + B_BYTES, &map_b_lo, kb * BK, item * T + n0, &full[s]);
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer (one thread) =====
        if (lane == 0) {
            uint32_t it = 0, tile_iter = 0;
            for (int tile = blockIdx.x; tile < tiles_total; tile += gridDim.x, ++tile_iter) {
                const uint32_t acc = tile_iter & 1;
                mbar_wait(&acc_empty[acc], ((tile_iter >> 1) & 1) ^ 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t tmem_d = tmem_base + acc * BN;
                for (int kb = 0; kb < KBLOCKS; ++kb, ++it) {
                    const int s = it % STAGES;
                    mbar_wait(&full[s], (it / STAGES) & 1);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const unsigned char* a_tile = tiles + (size_t)s * STAGE_BYTES;
                    const uint64_t da = umma_desc(a_tile), db = umma_desc(a_tile + A_BYTES);
#pragma unroll
                    for (int k = 0; k < BK / 8; ++k)  // 8 floats = 32 bytes = 2 descriptor units per K step
                        umma_tf32(tmem_d, da + 2 * k, db + 2 * k, Cfg::IDESC, (kb | k) ? 1u : 0u);
                    if (SPLIT3) {
                        const uint64_t da_lo = umma_desc(a_tile + A_BYTES + B_BYTES);
                        const uint64_t db_lo = umma_desc(a_tile + 2 * A_BYTES + B_BYTES);
#pragma unroll
                        for (int k = 0; k < BK / 8; ++k) {
                            umma_tf32(tmem_d, da + 2 * k, db_lo + 2 * k, Cfg::IDESC, 1u);  // hi lo^T
                            umma_tf32(tmem_d, da_lo + 2 * k, db + 2 * k, Cfg::IDESC, 1u);  // lo hi^T
                        }
                    }
                    umma_commit(&empty[s]);  // frees the stage once the MMAs have read it
                }
                umma_commit(&acc_full[acc]);  // accumulator complete
            }
        }
    } else {
        // ===== epilogue warps 2..5: TMEM lane quarter = warp % 4 =====
        const int quarter = warp & 3;
        float* stage = epi + quarter * 32 * EPI_PITCH;
        uint32_t tile_iter = 0;
        for (int tile = blockIdx.x; tile < tiles_total; tile += gridDim.x, ++tile_iter) {
            int item, mi, ni;
            decode_tile<TRI, Q>(tile, per_item, mt, nt, col_raster, item, mi, ni);
            const int m0 = r0 + mi * BM, n0 = ni * BN;
            // every element of S is written exactly once: (row, col) with col >= row directly, its mirror image
            // from the same registers; the part of a diagonal-crossing tile below the diagonal is dropped
            const bool crosses = TRI && n0 < m0 + BM;  // the tile holds elements on or below the diagonal
            const bool mirror = TRI && n0 + BN > m0 + 1;
            const uint32_t acc = tile_iter & 1;
            mbar_wait(&acc_full[acc], (tile_iter >> 1) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            float* __restrict__ Sitem = S + (size_t)item * rows * T;  // row-major rows [r0, row_end), pitch T
            const int row_base = m0 + quarter * 32;
#pragma unroll 1
            for (int chunk = 0; chunk < BN / 32; ++chunk) {
                uint32_t v[32];
                tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * BN + chunk * 32, v);
                // thread = row, v = 32 consecutive columns  ->  smem [row][col], read back [col] per row
#pragma unroll
                for (int c = 0; c < 32; ++c) stage[lane * EPI_PITCH + c] = __uint_as_float(v[c]);
                if (mirror && row_base + lane < T) {
                    // S[col][row] = S[row][col]: for a fixed column the 32 lanes hold 32 consecutive rows, so the
                    // mirrored tile goes out as 128-byte rows straight from the registers
                    float* __restrict__ dst = Sitem + (size_t)(n0 + chunk * 32) * T + row_base + lane;
                    const int above = row_base + lane - (n0 + chunk * 32);  // column offsets > above lie above the diagonal
#pragma unroll
                    for (int c = 0; c < 32; ++c)
                        if (n0 + chunk * 32 + c < T && (!crosses || c > above)) dst[(size_t)c * T] = __uint_as_float(v[c]);
                }
                __syncwarp();
                const int col = n0 + chunk * 32 + lane;
                if (col < T) {
#pragma unroll 4
                    for (int r = 0; r < 32; ++r) {
                        const int row = row_base + r;
                        if (row < row_end && (!crosses || col >= row)) Sitem[(size_t)(row - r0) * T + col] = stage[r * EPI_PITCH + lane];
                    }
                }
                __syncwarp();
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            if (lane == 0) mbar_arrive(&acc_empty[acc]);
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

bool make_map(CUtensorMap* map, const float* base, size_t rows, int box_rows) {
    EncodeTiledFn fn = encode_tiled();
    if (!fn) return false;
    const cuuint64_t dims[2] = {(cuuint64_t)KPAD, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)KPAD * sizeof(float)};
    const cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
    const cuuint32_t elem[2] = {1, 1};
    return fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, elem,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <int BN, bool SPLIT3, bool TRI>
int launch_gemm(cudaStream_t st, const float* hi, const float* lo, int n_items, int T, int r0, int rows, float* S,
                int sm_count) {
    using Cfg = GemmCfg<BN, SPLIT3>;
    CUtensorMap map_a, map_b, map_a_lo, map_b_lo;
    const size_t op_rows = (size_t)n_items * T;
    if (!make_map(&map_a, hi, op_rows, BM) || !make_map(&map_b, hi, op_rows, BN)) return -1;
    if (!make_map(&map_a_lo, SPLIT3 ? lo : hi, op_rows, BM) || !make_map(&map_b_lo, SPLIT3 ? lo : hi, op_rows, BN)) return -1;
    static SmemOptIn opt_in;
    {
        if (!smem_opt_in(k_simgemm<BN, SPLIT3, TRI>, (size_t)Cfg::SMEM, opt_in)) return -2;
    }
    const int mt = (rows + BM - 1) / BM, nt = (T + BN - 1) / BN;
    const int per_item = TRI ? triangle_tiles<BN / BM>(mt, nt) : mt * nt;
    const int tiles_total = n_items * per_item;
    const int grid = std::max(1, std::min(tiles_total, sm_count));
    const int col_raster = rows < T ? 1 : 0;
    k_simgemm<BN, SPLIT3, TRI><<<grid, GEMM_THREADS, Cfg::SMEM, st>>>(map_a, map_b, map_a_lo, map_b_lo, T, r0, rows, n_items,
                                                                      per_item, col_raster, S);
    return 0;
}

}  // namespace

// S[item] = A[item] A[item]^T for n_items stacked [T][KPAD] operands.  `lo` = nullptr: single TF32 pass
// on `hi`; otherwise the 3xTF32 split product of hi + lo.  Returns 0 on success.
int launch_selfsim_tc(cudaStream_t st, const float* hi, const float* lo, int n_items, int T, float* S, int sm_count) {
    // split product: 128 x 256 tiles (65 flop per operand byte from L2 instead of 49: the kernel runs at the L2
    // throughput cap, ncu profiles/r2a_sim); "simgemm_bn" = 128 selects the round-1 square tiles
    if (lo) {
        if (g_tuning.simgemm_bn == 128) return launch_gemm<128, true, true>(st, hi, lo, n_items, T, 0, T, S, sm_count);
        return launch_gemm<256, true, true>(st, hi, lo, n_items, T, 0, T, S, sm_count);
    }
    return launch_gemm<256, false, false>(st, hi, nullptr, n_items, T, 0, T, S, sm_count);
}

// Row panel of one item: S_panel[r - r0][c] = <A[r], A[c]> for r in [r0, r0 + rows), c < T, row-major with pitch T.
// The panel is a full rectangle (no mirror writes: S is not kept for later panels), so the split product costs twice
// the MMAs per element of the triangle.  Tiles are rastered column by column.
int launch_selfsim_tc_panel(cudaStream_t st, const float* hi, const float* lo, int T, int r0, int rows, float* S_panel,
                            int sm_count) {
    if (lo) {
        if (g_tuning.simgemm_bn == 128) return launch_gemm<128, true, false>(st, hi, lo, 1, T, r0, rows, S_panel, sm_count);
        return launch_gemm<256, true, false>(st, hi, lo, 1, T, r0, rows, S_panel, sm_count);
    }
    return launch_gemm<256, false, false>(st, hi, nullptr, 1, T, r0, rows, S_panel, sm_count);
}

}  // namespace repet
