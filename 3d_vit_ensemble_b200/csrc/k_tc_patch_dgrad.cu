// tcgen05 data gradient of the patch embedding (a1 backward w.r.t. the input volume), TF32, sm_100a:
//
//   dx[b,0, px*p0+i, py*p1+j, z] = sum_h dtokens[b, 1+p, h] * W[h, (i*p1+j)*p2+z]      (p = px*ny + py)
//
// Conv3d with stride == kernel has no overlapping patches, so this is one GEMM followed by a pure permutation - the
// inverse of the TMA im2col of the forward (k_tc_gemm.cu).  Both ends of the permutation are done by the TMA unit:
//   A  the patch rows of dtokens, read in place by a 3-D box {32 floats, P rows from row 1, 128/P volumes}: a tile
//      holds whole volumes and skips their cls rows;
//   B  the TF32-rounded transposed filter bank [Kp, H] viewed [H][inner = p1*p2][p0]: a 32-row chunk of the padded
//      N dimension (p0 x ceil(inner/32) x 32) belongs to ONE patch row i, zero-filled past the row end;
//   D  each 128 x 32 fp32 accumulator chunk is staged in shared memory and stored by the forward's own 5-D view of
//      the volume, box {32, ny, 1, nx, 128/P} at {c0, 0, i, 0, v0}; the out-of-bounds tail of a row is not written.
// The product is bound by the HBM write of dx (4 bytes per voxel); the filter bank is stationary in shared memory
// (one 128-column n-tile per CTA for its lifetime, at most 128 KB for H <= 256), so only the 128 KB A tiles stream.
//
//   warp 0: TMA producer    warp 1: TMEM allocator + MMA issuer    warps 2-5: epilogue (one TMEM lane quarter each)
#include "ptx.cuh"
#include "tc.cuh"
#include "tc_epilogue.cuh"

namespace vit3d {

using namespace ptx;

namespace {

constexpr int DG_BM = 128;                          // token rows per tile
constexpr int DG_BN = 128;                          // padded output columns per tile (four 32-column chunks)
constexpr int DG_CHUNKS = DG_BN / 32;
constexpr int DG_MAX_H = 256;
constexpr int DG_A_BYTES = DG_BM * 128;             // one k-block of A: 128 rows x 32 floats
constexpr int DG_BKB_BYTES = DG_BN * 128;           // one k-block of the filter slab
constexpr int DG_SLAB_BYTES = (DG_MAX_H / 32) * DG_BKB_BYTES;
constexpr int DG_STAGES = 4;
constexpr int DG_STG_BYTES = DG_BM * 128;           // one staged 128 x 32 fp32 output chunk
constexpr int DG_THREADS = 192;
constexpr int DG_SMEM_BYTES = DG_SLAB_BYTES + DG_STAGES * DG_A_BYTES + 2 * DG_STG_BYTES + 256;
static_assert(DG_SMEM_BYTES <= 232448, "over the 227 KB shared-memory limit");

__device__ __forceinline__ void tma_store_5d(const CUtensorMap* m, uint32_t smem_src, int c0, int c1, int c2, int c3, int c4) {
  asm volatile("cp.async.bulk.tensor.5d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5, %6}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_src), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
               : "memory");
}
// all but the most recent bulk store group have finished reading shared memory
__device__ __forceinline__ void bulk_store_wait_read_1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }

__global__ void __launch_bounds__(DG_THREADS, 1)
tc_patch_dgrad_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                      const __grid_constant__ CUtensorMap tmD, int nkb, int tiles_m, int tiles_n, int nch, int p0, int vpt) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* slab = smem_raw;                          // 128B-swizzled operand tiles need 1024-byte alignment
  if (smem_u32(slab) & 1023u) __trap();
  uint8_t* ring = slab + DG_SLAB_BYTES;
  uint8_t* stg = ring + DG_STAGES * DG_A_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(stg + 2 * DG_STG_BYTES);
  uint64_t* full_bar = bars;                         // [DG_STAGES]
  uint64_t* empty_bar = bars + DG_STAGES;            // [DG_STAGES]
  uint64_t* tmem_full = bars + 2 * DG_STAGES;        // [2]
  uint64_t* tmem_empty = bars + 2 * DG_STAGES + 2;   // [2]
  uint64_t* slab_full = bars + 2 * DG_STAGES + 4;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 2 * DG_STAGES + 5);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  // stationary schedule: the CTA keeps n-tile tn and walks the row tiles tm0, tm0 + cpn, ...
  const int tn = blockIdx.x % tiles_n, tm0 = blockIdx.x / tiles_n, cpn = gridDim.x / tiles_n;
  const int total_chunks = p0 * nch;
  const int nvalid = min(DG_CHUNKS, total_chunks - tn * DG_CHUNKS);

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    prefetch_tmap(&tmD);
    for (int s = 0; s < DG_STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tmem_full[b], 1);
      mbar_init(&tmem_empty[b], 4);                  // one arrival per epilogue warp
    }
    mbar_init(slab_full, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<2 * DG_BN>(tmem_ptr_smem);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  pdl_trigger();
  pdl_wait();

  if (warp == 0) {
    // ===================================================== TMA producer
    if (lane == 0) {
      // the n-tile's filter chunks, once: chunk ch of k-block kb at slab + kb * 16 KB + ch * 4 KB (rows of 128 B)
      mbar_arrive_expect_tx(slab_full, nkb * nvalid * 32 * 128);
      for (int kb = 0; kb < nkb; ++kb)
        for (int ch = 0; ch < nvalid; ++ch) {
          const int g = tn * DG_CHUNKS + ch;
          tma_load_3d(slab + kb * DG_BKB_BYTES + ch * 32 * 128, &tmB, slab_full, kb * 32, (g % nch) * 32, g / nch);
        }
      int stage = 0;
      uint32_t phase = 0;
      for (int tm = tm0; tm < tiles_m; tm += cpn)
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          mbar_arrive_expect_tx(&full_bar[stage], DG_A_BYTES);
          tma_load_3d(ring + stage * DG_A_BYTES, &tmA, &full_bar[stage], kb * 32, 1, tm * vpt);
          if (++stage == DG_STAGES) { stage = 0; phase ^= 1; }
        }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================================================== MMA issuer (one thread for the whole schedule)
    if (elect_one()) {
      const uint32_t idesc = make_idesc(UMMA_FMT_TF32, DG_BM, DG_BN, 0, 0);
      const uint64_t ring_desc = make_smem_desc(smem_u32(ring), 16, 1024, UMMA_LAYOUT_SW128);
      const uint64_t slab_desc = make_smem_desc(smem_u32(slab), 16, 1024, UMMA_LAYOUT_SW128);
      mbar_wait(slab_full, 0);
      int stage = 0, it = 0;
      uint32_t phase = 0;
      for (int tm = tm0; tm < tiles_m; tm += cpn, ++it) {
        const int buf = it & 1;
        mbar_wait(&tmem_empty[buf], ((it >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + buf * DG_BN;
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          const uint64_t ad = ring_desc + (uint64_t)((stage * DG_A_BYTES) >> 4);
          const uint64_t bd = slab_desc + (uint64_t)((kb * DG_BKB_BYTES) >> 4);
#pragma unroll
          for (int k = 0; k < 4; ++k)      // 4 x 32 bytes of K (8 tf32) per k-block
            umma<true>(d_tmem, ad + 2 * k, bd + 2 * k, idesc, (kb > 0 || k > 0) ? 1u : 0u);
          umma_commit(&empty_bar[stage]);
          if (++stage == DG_STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tmem_full[buf]);
      }
    }
    __syncwarp();
  } else {
    // ===================================================== epilogue: TMEM -> swizzled staging chunk -> 5-D TMA store
    const int q = warp & 3;                          // the TMEM lane quarter this warp may read
    const int row = q * 32 + lane;                   // tile row = (volume, px, py), the order of the store box
    const bool issuer = threadIdx.x == 64;
    int nst = 0;
    int it = 0;
    for (int tm = tm0; tm < tiles_m; tm += cpn, ++it) {
      const int buf = it & 1;
      mbar_wait(&tmem_full[buf], (it >> 1) & 1);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + buf * DG_BN;
      for (int ch = 0; ch < nvalid; ++ch, ++nst) {
        uint32_t r[32];
        tmem_ld_32x32b_x32(taddr + ch * 32, r);
        const uint32_t sb = smem_u32(stg + (nst & 1) * DG_STG_BYTES);
        if (issuer) bulk_store_wait_read_1();        // the store that last read this staging buffer is done with it
        tmem_ld_wait();
        if (ch == nvalid - 1) {                      // the accumulator is in registers: the next tile may start
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&tmem_empty[buf]);
        }
        asm volatile("bar.sync 1, 128;" ::: "memory");
        const uint32_t my_row = sb + row * 128;
#pragma unroll
        for (int j = 0; j < 8; ++j)
          st_shared_v4(my_row + ((j ^ (row & 7)) << 4), r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
        fence_proxy_async_smem();
        asm volatile("bar.sync 1, 128;" ::: "memory");
        if (issuer) {
          const int g = tn * DG_CHUNKS + ch;
          tma_store_5d(&tmD, sb, (g % nch) * 32, 0, g / nch, 0, tm * vpt);
          bulk_store_commit();
        }
      }
    }
    if (issuer) bulk_store_wait_all();               // bulk tensor stores must complete before the CTA exits
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc<2 * DG_BN>(tmem_base);
}

}  // namespace

bool tc_patch_dgrad_supported(int B, int X, int Y, int Z, int p0, int p1, int p2, int H) {
  if (!tc_patch_embed_supported(B, X, Y, Z, p0, p1, p2, H) || H > DG_MAX_H) return false;
  const int nch = ceil_div(p1 * p2, 32);
  return ceil_div(p0 * nch, DG_CHUNKS) <= sm_count();
}

int tc_patch_dgrad(const float* dtokens, const float* w_t, float* dx, int B, int X, int Y, int Z, int p0, int p1, int p2,
                   int H, cudaStream_t st) {
  if (!tc_patch_dgrad_supported(B, X, Y, Z, p0, p1, p2, H)) V3_UNSUPPORTED("tc patch dgrad: unsupported geometry");
  const int nx = X / p0, ny = Y / p1, P = nx * ny, S = P + 1, inner = p1 * p2;
  const int vpt = DG_BM / P;
  const int nch = ceil_div(inner, 32);
  const int tiles_m = ceil_div(B, vpt), tiles_n = ceil_div(p0 * nch, DG_CHUNKS);
  CUtensorMap ta, tb, td;
  {
    // dtokens viewed (innermost first): [H][S tokens][B volumes]; the box starts at token 1 (the cls rows are skipped)
    cuuint64_t dims[3] = {(cuuint64_t)H, (cuuint64_t)S, (cuuint64_t)B};
    cuuint64_t str[2] = {(cuuint64_t)H * 4, (cuuint64_t)S * H * 4};
    cuuint32_t box[3] = {32, (cuuint32_t)P, (cuuint32_t)vpt};
    int rc = make_tmap_nd(&ta, dtokens, 3, dims, str, box);
    if (rc != VIT3D_OK) return rc;
    // w_t [Kp, H] viewed: [H][inner][p0]
    cuuint64_t wd[3] = {(cuuint64_t)H, (cuuint64_t)inner, (cuuint64_t)p0};
    cuuint64_t wstr[2] = {(cuuint64_t)H * 4, (cuuint64_t)inner * H * 4};
    cuuint32_t wb[3] = {32, 32, 1};
    rc = make_tmap_nd(&tb, w_t, 3, wd, wstr, wb);
    if (rc != VIT3D_OK) return rc;
    // dx viewed exactly as the forward views x: [inner floats][ny patches][p0 rows][nx patches][B volumes]
    cuuint64_t xd[5] = {(cuuint64_t)inner, (cuuint64_t)ny, (cuuint64_t)p0, (cuuint64_t)nx, (cuuint64_t)B};
    cuuint64_t xs[4] = {(cuuint64_t)inner * 4, (cuuint64_t)Y * Z * 4, (cuuint64_t)p0 * Y * Z * 4, (cuuint64_t)X * Y * Z * 4};
    cuuint32_t xb[5] = {32, (cuuint32_t)ny, 1, (cuuint32_t)nx, (cuuint32_t)vpt};
    rc = make_tmap_nd(&td, dx, 5, xd, xs, xb);
    if (rc != VIT3D_OK) return rc;
  }
  static thread_local int configured_dev = -1;
  int dev = 0;
  V3_CUDA(cudaGetDevice(&dev));
  if (configured_dev != dev) {
    V3_CUDA(cudaFuncSetAttribute(tc_patch_dgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, DG_SMEM_BYTES));
    configured_dev = dev;
  }
  int cpn = sm_count() / tiles_n;                    // CTAs per n-tile
  if (cpn > tiles_m) cpn = tiles_m;
  V3_CUDA(launch_pdl(tc_patch_dgrad_kernel, dim3(cpn * tiles_n), dim3(DG_THREADS), (size_t)DG_SMEM_BYTES, st, ta, tb, td,
                     H / 32, tiles_m, tiles_n, nch, p0, vpt));
  V3_LAUNCH_CHECK();
  return VIT3D_OK;
}

}  // namespace vit3d
