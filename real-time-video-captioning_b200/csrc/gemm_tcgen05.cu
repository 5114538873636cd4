// Persistent warp-specialised bf16 GEMM for sm_100a:  C = act(A * W^T + bias) + residual.
//
//   * operands A [M,K] and W [N,K] (both K-major) are brought into shared memory by TMA
//     (cp.async.bulk.tensor, 128-byte swizzle) through a multi-stage mbarrier ring,
//   * one elected thread issues tcgen05.mma (kind::f16, M=128, N=BN, K=16) with the fp32 accumulator
//     in TMEM; two accumulator buffers let the epilogue of tile i overlap the MMAs of tile i+1,
//   * four epilogue warps read the accumulator back with tcgen05.ld and apply the fused epilogue
//     (bias, QuickGELU / erf-GELU, residual or positional-embedding add, bf16 and/or fp32 store).
//
// This one kernel covers every dense contraction of the captioning path (SURVEY.md §2.3 K1, K3, K7,
// K9, K12): patch embedding, ViT QKV / out-proj / MLP, visual projection, decoder QKV / out / FFN and
// the vocabulary head.
#include <cuda.h>

#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "common.cuh"
#include "kernels.h"

cudaError_t gemm2_bf16(const GemmArgs& a, cudaStream_t stream);
cudaError_t gemv_skinny(const GemmArgs& a, cudaStream_t stream);

namespace {

constexpr int BM = 128;       // rows per tile = UMMA M = TMEM lanes
constexpr int BK = 64;        // K elements per pipeline stage = one 128-byte swizzle row of bf16
constexpr int UMMA_K = 16;    // K per tcgen05.mma for 16-bit inputs
constexpr int NUM_EPI_WARPS = 8;  // two warps per TMEM lane quarter, each owning half of the tile's columns
constexpr int NUM_THREADS = 64 + 32 * NUM_EPI_WARPS;  // warp 0: TMA producer, warp 1: MMA issuer + TMEM owner, warps 2-9: epilogue
constexpr int SMEM_BUDGET = 200 * 1024;

template <int BN>
struct Cfg {
  static constexpr int A_BYTES = BM * BK * 2;
  static constexpr int B_BYTES = BN * BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES = SMEM_BUDGET / STAGE_BYTES;  // 4 for BN=256, 6 for BN=128
  static constexpr int TMEM_COLS = 2 * BN;                  // two accumulator buffers
  static constexpr int F32_STAGE_BYTES = NUM_EPI_WARPS * 32 * 32 * 4;  // fp32 output: one 32 x 32 transpose slice per epilogue warp
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/ + F32_STAGE_BYTES;
};

struct Epilogue {
  const float* bias;
  const bf16* residual;
  int ldr;
  int res_periodic;
  int act;
  bf16* out;
  int ldo;
  float* out_f32;
  int ldo32;
  int gin, gout, goff;
};

template <int BN>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b, int M,
                    int N, int K, Epilogue ep) {
  using C = Cfg<BN>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = ptx::warp_uniform((ptx::smem_u32(smem_raw) + 1023u) & ~1023u);  // SWIZZLE_128B wants 1024-B alignment
  const uint32_t bar_base = smem_base + C::STAGES * C::STAGE_BYTES;
  // barrier block: full[STAGES] | empty[STAGES] | tmem_full[2] | tmem_empty[2] | tmem base address
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (C::STAGES + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * C::STAGES + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * C::STAGES + 2 + a); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * C::STAGES + 4);
  float* const f32_stage = reinterpret_cast<float*>(smem_raw + (smem_base - ptx::smem_u32(smem_raw)) + C::STAGES * C::STAGE_BYTES + 256);
  auto smem_a = [&](int s) { return smem_base + s * C::STAGE_BYTES; };
  auto smem_b = [&](int s) { return smem_base + s * C::STAGE_BYTES + C::A_BYTES; };

  const int warp = __shfl_sync(0xffffffffu, (int)threadIdx.x / 32, 0);
  const int lane = threadIdx.x & 31;

  const int m_tiles = (M + BM - 1) / BM;
  const int n_tiles = N / BN;
  const int num_tiles = m_tiles * n_tiles;
  const int num_kb = (K + BK - 1) / BK;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&tmap_a);
    ptx::prefetch_tensormap(&tmap_b);
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < C::STAGES; ++s) {
        ptx::mbar_init(full_bar(s), 1);
        ptx::mbar_init(empty_bar(s), 1);
      }
      for (int a = 0; a < 2; ++a) {
        ptx::mbar_init(tfull_bar(a), 1);
        ptx::mbar_init(tempty_bar(a), NUM_EPI_WARPS);  // one arrival per epilogue warp
      }
      ptx::fence_barrier_init();
    }
    __syncwarp();
    ptx::tmem_alloc(tmem_slot, C::TMEM_COLS);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
  tmem_base = ptx::warp_uniform(tmem_base);

  // Producer and MMA issuer run as WHOLE warps in warp-uniform control flow; one elected lane executes each TMA /
  // tcgen05 instruction (common.cuh: issuing from an `if (lane == 0)` region makes ptxas wrap every UTCHMMA in a
  // ~25-instruction waterfall loop).
  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int m0 = (tile / n_tiles) * BM;
        const int n0 = (tile % n_tiles) * BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          ptx::mbar_wait(empty_bar(stage), phase ^ 1u);
          ptx::mbar_arrive_expect_tx_elect(full_bar(stage), C::STAGE_BYTES);
          ptx::tma_load_2d_elect(smem_a(stage), &tmap_a, full_bar(stage), kb * BK, m0);
          ptx::tma_load_2d_elect(smem_b(stage), &tmap_b, full_bar(stage), kb * BK, n0);
          if (++stage == C::STAGES) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer (whole warp, elected lane issues)
    {
      constexpr uint32_t idesc = ptx::umma_idesc_bf16(BM, BN);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        ptx::mbar_wait(tempty_bar(acc), acc_phase ^ 1u);  // epilogue has drained this accumulator
        ptx::tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
        for (int kb = 0; kb < num_kb; ++kb) {
          ptx::mbar_wait(full_bar(stage), phase);  // TMA bytes have landed
          ptx::tc_fence_after();
          const uint64_t da = ptx::umma_desc_sw128_kmajor(smem_a(stage));
          const uint64_t db = ptx::umma_desc_sw128_kmajor(smem_b(stage));
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) {
            // advancing K by 16 bf16 = 32 bytes inside the 128-byte swizzle row: +2 in the (addr >> 4) field
            ptx::umma_bf16_elect(d_tmem, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (kb | k) != 0);
          }
          ptx::umma_commit_elect(empty_bar(stage));  // smem slot is free once these MMAs have read it
          if (kb == num_kb - 1) ptx::umma_commit_elect(tfull_bar(acc));  // accumulator complete
          if (++stage == C::STAGES) {
            stage = 0;
            phase ^= 1u;
          }
        }
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1u;
      }
    }
  } else {
    // ------------------------------------------------------------ epilogue warps (TMEM -> regs -> global)
    const int quarter = warp & 3;  // a warp may only touch TMEM lanes [32*(warp%4), +32)
    const int c_begin = ((warp - 2) >> 2) * (BN / 2);  // warps 2-5: left half of the columns, 6-9: right half
    const int c_end = c_begin + BN / 2;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const int m0 = (tile / n_tiles) * BM;
      const int n0 = (tile % n_tiles) * BN;
      ptx::mbar_wait(tfull_bar(acc), acc_phase);
      ptx::tc_fence_after();
      const int r = m0 + quarter * 32 + lane;
      const bool row_ok = r < M;
      int orow = r;
      int rrow = r;
      if (ep.gin > 0) {
        orow = (r / ep.gin) * ep.gout + (r % ep.gin) + ep.goff;
        rrow = ep.res_periodic ? (r % ep.gin) + ep.goff : orow;
      }
      const uint32_t t_row = tmem_base + (uint32_t)(acc * BN) + ((uint32_t)(quarter * 32) << 16);
#pragma unroll 1
      for (int c = c_begin; c < c_end; c += 32) {
        uint32_t v[32];
        ptx::tmem_ld_32x32b_x32(t_row + (uint32_t)c, v);
        ptx::tmem_ld_wait();
        const int col = n0 + c;
        float f[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) f[i] = __uint_as_float(v[i]);
        if (row_ok) {
          if (ep.bias != nullptr) {
            const float4* b4 = reinterpret_cast<const float4*>(ep.bias + col);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float4 b = __ldg(b4 + i);
              f[4 * i + 0] += b.x;
              f[4 * i + 1] += b.y;
              f[4 * i + 2] += b.z;
              f[4 * i + 3] += b.w;
            }
          }
          if (ep.act == ACT_QUICK_GELU) {
#pragma unroll
            for (int i = 0; i < 32; ++i) f[i] = quick_gelu(f[i]);
          } else if (ep.act == ACT_GELU_ERF) {
#pragma unroll
            for (int i = 0; i < 32; ++i) f[i] = gelu_erf(f[i]);
          } else if (ep.act == ACT_RELU) {
#pragma unroll
            for (int i = 0; i < 32; ++i) f[i] = fmaxf(f[i], 0.f);
          }
          if (ep.residual != nullptr) {
            const uint4* r4 = reinterpret_cast<const uint4*>(ep.residual + (size_t)rrow * ep.ldr + col);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const uint4 u = r4[i];  // plain load: `out` may alias `residual` (in-place residual update)
              const float2 a0 = unpack_bf16(u.x), a1 = unpack_bf16(u.y), a2 = unpack_bf16(u.z), a3 = unpack_bf16(u.w);
              f[8 * i + 0] += a0.x;
              f[8 * i + 1] += a0.y;
              f[8 * i + 2] += a1.x;
              f[8 * i + 3] += a1.y;
              f[8 * i + 4] += a2.x;
              f[8 * i + 5] += a2.y;
              f[8 * i + 6] += a3.x;
              f[8 * i + 7] += a3.y;
            }
          }
          if (ep.out != nullptr) {
            uint4* o4 = reinterpret_cast<uint4*>(ep.out + (size_t)orow * ep.ldo + col);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              uint4 u;
              u.x = pack_bf16(f[8 * i + 0], f[8 * i + 1]);
              u.y = pack_bf16(f[8 * i + 2], f[8 * i + 3]);
              u.z = pack_bf16(f[8 * i + 4], f[8 * i + 5]);
              u.w = pack_bf16(f[8 * i + 6], f[8 * i + 7]);
              o4[i] = u;
            }
          }
        }
        if (ep.out_f32 != nullptr) {  // warp-uniform
          // A lane holds 32 consecutive columns of ONE row: stored directly, every instruction would touch 32 rows with 16 bytes
          // each (half-written sectors: the vocabulary head ran at 1.1 TB/s of logits).  The 32 x 32 block goes through this warp's
          // shared-memory slice (16-byte chunk index XOR row: conflict-free both ways) and leaves as whole 128-byte row segments,
          // four rows per instruction.
          float* st = f32_stage + (warp - 2) * 1024;
#pragma unroll
          for (int i = 0; i < 8; ++i)
            *reinterpret_cast<float4*>(st + lane * 32 + ((i ^ (lane & 7)) << 2)) = make_float4(f[4 * i], f[4 * i + 1], f[4 * i + 2], f[4 * i + 3]);
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int rr = j * 4 + (lane >> 3), ch = lane & 7;
            const float4 val = *reinterpret_cast<const float4*>(st + rr * 32 + ((ch ^ (rr & 7)) << 2));
            const int r2 = m0 + quarter * 32 + rr;
            if (r2 < M) {
              const int o2 = ep.gin > 0 ? (r2 / ep.gin) * ep.gout + (r2 % ep.gin) + ep.goff : r2;
              *reinterpret_cast<float4*>(ep.out_f32 + (size_t)o2 * ep.ldo32 + col + ch * 4) = val;
            }
          }
          __syncwarp();
        }
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(tempty_bar(acc));
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1u;
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, C::TMEM_COLS);
  }
}

// ------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

std::string g_err;
std::mutex g_mu;

EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn == nullptr) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

struct MapKey {
  const void* ptr;
  int rows, cols, ld, box_rows, box_cols;
  bool operator==(const MapKey& o) const {
    return ptr == o.ptr && rows == o.rows && cols == o.cols && ld == o.ld && box_rows == o.box_rows && box_cols == o.box_cols;
  }
};
struct MapKeyHash {
  size_t operator()(const MapKey& k) const {
    size_t h = reinterpret_cast<size_t>(k.ptr);
    h = h * 1000003u ^ (size_t)k.rows;
    h = h * 1000003u ^ (size_t)k.cols;
    h = h * 1000003u ^ (size_t)k.ld;
    h = h * 1000003u ^ (size_t)k.box_rows;
    h = h * 1000003u ^ (size_t)k.box_cols;
    return h;
  }
};
std::unordered_map<MapKey, CUtensorMap, MapKeyHash> g_maps;

}  // namespace

// 2-D bf16 tensor map over a row-major [rows, cols] matrix (leading dimension ld), box = box_cols x box_rows
// (box_cols * 2 bytes == 128), 128-byte swizzle; out-of-bounds elements read as zero / are not written (M, K tails).
bool gemm_get_tensor_map(const bf16* ptr, int rows, int cols, int ld, int box_cols, int box_rows, CUtensorMap* out) {
  MapKey key{ptr, rows, cols, ld, box_rows, box_cols};
  std::lock_guard<std::mutex> lk(g_mu);
  auto it = g_maps.find(key);
  if (it != g_maps.end()) {
    *out = it->second;
    return true;
  }
  EncodeTiledFn fn = encode_fn();
  if (fn == nullptr) {
    g_err = "cuTensorMapEncodeTiled entry point not available (no CUDA driver?)";
    return false;
  }
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstride[1] = {(cuuint64_t)ld * sizeof(bf16)};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  cuuint32_t estride[2] = {1, 1};
  CUtensorMap m;
  CUresult r = fn(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<bf16*>(ptr), gdim, gstride, box, estride,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    g_err = "cuTensorMapEncodeTiled failed with CUresult " + std::to_string((int)r);
    return false;
  }
  if (g_maps.size() > 4096) g_maps.clear();
  g_maps.emplace(key, m);
  *out = m;
  return true;
}

int gemm_sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

namespace {

template <int BN>
cudaError_t launch(const GemmArgs& a, const Epilogue& ep, cudaStream_t stream) {
  using C = Cfg<BN>;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e =
        cudaFuncSetAttribute(gemm_tcgen05_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES);
    if (e != cudaSuccess) return e;
    attr_set = true;
  }
  CUtensorMap ta, tb;
  if (!gemm_get_tensor_map(a.A, a.M, a.K, a.lda, BK, BM, &ta)) return cudaErrorInvalidValue;
  if (!gemm_get_tensor_map(a.W, a.N, a.K, a.ldw, BK, BN, &tb)) return cudaErrorInvalidValue;
  const int tiles = ((a.M + BM - 1) / BM) * (a.N / BN);
  const int grid = tiles < gemm_sm_count() ? tiles : gemm_sm_count();
  gemm_tcgen05_kernel<BN><<<grid, NUM_THREADS, C::SMEM_BYTES, stream>>>(ta, tb, a.M, a.N, a.K, ep);
  note_launch();
  return cudaGetLastError();
}

// ---- optional per-launch timing with CUDA events on the launching stream (bench.py's roofline leg)
struct Prof {
  bool on = false;
  std::vector<cudaEvent_t> ev;  // pairs
  std::vector<double> flops;
  size_t used = 0;              // pairs in flight
  double ms = 0, fl = 0;
  long long n = 0;
} g_prof;

void prof_drain() {
  for (size_t i = 0; i < g_prof.used; ++i) {
    cudaEventSynchronize(g_prof.ev[2 * i + 1]);
    float t = 0;
    if (cudaEventElapsedTime(&t, g_prof.ev[2 * i], g_prof.ev[2 * i + 1]) == cudaSuccess) {
      g_prof.ms += t;
      g_prof.fl += g_prof.flops[i];
      ++g_prof.n;
    }
  }
  g_prof.used = 0;
}

}  // namespace

const char* gemm_last_error() { return g_err.c_str(); }

void gemm_profile_enable(int on) {
  if (on && g_prof.ev.empty()) {
    g_prof.ev.resize(2 * 8192);
    g_prof.flops.resize(8192);
    for (auto& e : g_prof.ev) cudaEventCreate(&e);
  }
  if (on) {
    g_prof.used = 0;
    g_prof.ms = g_prof.fl = 0;
    g_prof.n = 0;
  }
  g_prof.on = on != 0;
}

bool gemm_profile_enabled() { return g_prof.on; }

void gemm_profile_read(double* ms, double* flops, long long* launches) {
  prof_drain();
  *ms = g_prof.ms;
  *flops = g_prof.fl;
  *launches = g_prof.n;
}

cudaError_t gemm_bf16(const GemmArgs& a, cudaStream_t stream, int force_bn) {
  if (a.M <= 0) return cudaSuccess;
  if (a.N % 128 != 0 || a.K % 8 != 0 || a.lda % 8 != 0 || a.ldw % 8 != 0 || a.K <= 0 ||
      (a.out != nullptr && a.ldo % 8 != 0) || (a.out_f32 != nullptr && a.ldo32 % 4 != 0) ||
      (a.residual != nullptr && a.ldr % 8 != 0) || (a.out == nullptr && a.out_f32 == nullptr)) {
    g_err = "gemm_bf16: unsupported shape/stride (need N%128==0, K%8==0, 16-byte aligned rows)";
    return cudaErrorInvalidValue;
  }
  // checked here, not in gemv_skinny: a shape the skinny kernel declines would otherwise run on a tensor-core kernel WITHOUT the fusion
  if ((a.lnl_gamma != nullptr || a.sc_kv != nullptr) && (a.M > 8 || (force_bn != 0 && force_bn != 1) || a.gin > 0 || a.res_periodic)) {
    g_err = "gemm_bf16: LayerNorm-on-load / K-V scatter exist only in the skinny kernel (M <= 8)";
    return cudaErrorInvalidValue;
  }
  Epilogue ep{a.bias, a.residual, a.ldr, a.res_periodic, a.act, a.out, a.ldo, a.out_f32, a.ldo32, a.gin, a.gout, a.goff};
  int bn = force_bn;
  if (bn == 0) {
    const long tiles256 = (long)((a.M + BM - 1) / BM) * (a.N / 256);
    bn = (a.N % 256 == 0 && tiles256 >= gemm_sm_count()) ? 256 : 128;
    // large-M contractions go to the CTA-pair kernel (256x256 tiles, TMA-store epilogue) when its epilogue applies
    // ... unless the whole problem is one wave of 128 x 128 tiles (decode-step GEMMs at 1024-2048 rows: the pair kernel would keep
    // 24-72 of the 148 SMs busy; measured alone at M = 1024: 9.4 / 8.7 / 14.5 us against 11.5 / 11.2 / 21.6 us for QKV / out / fc2)
    const long tiles128 = (long)((a.M + BM - 1) / BM) * (a.N / 128);
    if (a.M >= 1024 && a.N % 256 == 0 && a.out != nullptr && a.out_f32 == nullptr && a.gin == 0 && !a.res_periodic) bn = 2;
    if (bn == 2 && tiles128 <= gemm_sm_count()) bn = 128;
  }
  size_t slot = 0;
  if (g_prof.on) {
    if (g_prof.used == g_prof.flops.size()) prof_drain();
    slot = g_prof.used++;
    g_prof.flops[slot] = 2.0 * a.M * a.N * a.K;
    cudaEventRecord(g_prof.ev[2 * slot], stream);
  }
  cudaError_t e = cudaErrorNotSupported;
  if (a.ln_stats != nullptr || a.stats_out != nullptr || a.lnout != nullptr) {  // only the CTA-pair kernel implements the folded / fused LayerNorm
    e = gemm2_bf16(a, stream);
    if (e == cudaErrorNotSupported) {
      g_err = "gemm_bf16: folded LayerNorm / row statistics need the CTA-pair kernel (N % 256 == 0, bf16 output, no remap)";
      e = cudaErrorInvalidValue;
    }
  } else if (force_bn == 1 || (force_bn == 0 && a.M <= 8)) e = gemv_skinny(a, stream);  // weight-streaming path for a few rows
  else if (bn == 2) e = gemm2_bf16(a, stream);
  if (e == cudaErrorNotSupported) e = (bn != 128 && a.N % 256 == 0) ? launch<256>(a, ep, stream) : launch<128>(a, ep, stream);
  if (g_prof.on) cudaEventRecord(g_prof.ev[2 * slot + 1], stream);
  return e;
}
