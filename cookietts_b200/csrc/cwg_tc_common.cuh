// Shared host/device helpers of the tensor-core kernels (cwg_tc.cu, cwg_wf.cu): tensor-map
// construction, UMMA issue helpers, TMEM load helpers, bf16 hi/lo split stores, the gate.
#pragma once

#include "cwg_common.cuh"
#include "cwg_sm100.cuh"

namespace cwg { namespace tc {

using namespace sm100;

// ------------------------------------------------------------------------------------------
// host: tensor maps (driver entry point resolved at run time; no link-time libcuda dependency)
// ------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                    CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                    CUtensorMapFloatOOBfill);

inline PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
      q != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = (PFN_encodeTiled)p;
  return fn;
}

// bf16 tensor, innermost dim contiguous, 128B swizzle, zero OOB fill. strides_bytes has rank-1 entries.
inline int make_map(CUtensorMap* m, const void* ptr, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
             const uint32_t* box, bool bytes = false, bool sw32 = false) {
  PFN_encodeTiled enc = get_encode();
  CWG_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t gd[5]; cuuint64_t gs[5]; cuuint32_t bx[5]; cuuint32_t es[5];
  for (int i = 0; i < rank; ++i) { gd[i] = dims[i]; bx[i] = box[i]; es[i] = 1; }
  for (int i = 0; i + 1 < rank; ++i) gs[i] = strides_bytes[i];
  CUresult r = enc(m, bytes ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(ptr), gd, gs, bx, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, sw32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  CWG_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
  return 0;
}

inline int map_2d(CUtensorMap* m, const void* ptr, uint64_t cols, uint64_t rows, uint32_t box_rows) {
  uint64_t dims[2] = {cols, rows}; uint64_t st[1] = {cols * 2}; uint32_t box[2] = {64, box_rows};
  return make_map(m, ptr, 2, dims, st, box);
}

// activations [B][T'][C] bf16 as (C, T', B); box = 64 channels x 128 steps of one utterance.
// Out-of-range steps (negative or >= T') are zero-filled: the conv's zero padding, per utterance.
inline int map_act(CUtensorMap* m, const void* ptr, uint64_t C, uint64_t Tp, uint64_t B) {
  uint64_t dims[3] = {C, Tp, B}; uint64_t st[2] = {C * 2, Tp * C * 2}; uint32_t box[3] = {64, 128, 1};
  return make_map(m, ptr, 3, dims, st, box);
}

// layer-0 fold (start conv folded into the in_layer): the coupling input planes [B][T'][16] 16-bit as (16, T', B), box = 16
// channels x 128 steps (4 KB, 32-byte rows, 32B swizzle), and the folded weights [rows][48] (3 taps x 16), box 16 x 128 rows
inline int map_a0(CUtensorMap* m, const void* ptr, uint64_t Tp, uint64_t B) {
  uint64_t dims[3] = {16, Tp, B}; uint64_t st[2] = {32, Tp * 32}; uint32_t box[3] = {16, 128, 1};
  return make_map(m, ptr, 3, dims, st, box, false, true);
}
inline int map_w0(CUtensorMap* m, const void* ptr, uint64_t rows) {
  uint64_t dims[2] = {48, rows}; uint64_t st[1] = {96}; uint32_t box[2] = {16, 128};
  return make_map(m, ptr, 2, dims, st, box, false, true);
}

// 8-bit (e5m2) planes: the same tiles measured in bytes - 128 channels x 128 steps / 128 k x box_rows rows = 16 KB units
inline int map_2d8(CUtensorMap* m, const void* ptr, uint64_t cols, uint64_t rows, uint32_t box_rows) {
  uint64_t dims[2] = {cols, rows}; uint64_t st[1] = {cols}; uint32_t box[2] = {128, box_rows};
  return make_map(m, ptr, 2, dims, st, box, true);
}
inline int map_act8(CUtensorMap* m, const void* ptr, uint64_t C, uint64_t Tp, uint64_t B) {
  uint64_t dims[3] = {C, Tp, B}; uint64_t st[2] = {C, Tp * C}; uint32_t box[3] = {128, 128, 1};
  return make_map(m, ptr, 3, dims, st, box, true);
}

// ------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------
constexpr int TILE_A = 128 * 128;      // [128 rows][64 bf16] = 16 KB
constexpr uint32_t IDESC_N256 = umma_idesc_bf16(128, 256);
constexpr uint32_t IDESC_N16 = umma_idesc_bf16(128, 16);
constexpr uint32_t IDESC_F16_N256 = umma_idesc_f16(128, 256);

__device__ __forceinline__ uint8_t* align_1024(uint8_t* p) {
  uint32_t a = smem_u32(p);
  return p + ((1024u - (a & 1023u)) & 1023u);
}

// One 64-deep k-block = 4 UMMA K-steps of 16 bf16 (32 bytes along the swizzled row).
__device__ __forceinline__ void issue_kblock(uint32_t a_addr, uint32_t b_addr, uint32_t tmem_d, uint32_t idesc, bool first) {
#pragma unroll
  for (int k = 0; k < 4; ++k)
    umma_bf16(tmem_d, umma_desc_sw128(a_addr + 32 * k), umma_desc_sw128(b_addr + 32 * k), idesc, (first && k == 0) ? 0u : 1u);
}

// 16-column TMEM load + wait in ONE asm block so no consumer can be scheduled before the wait
__device__ __forceinline__ void tmem_ld16_sync(uint32_t ta, float* a) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n\t"
      "tcgen05.wait::ld.sync.aligned;"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(ta)
      : "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) a[i] = __uint_as_float(r[i]);
}

// 16 fp32 values of one row -> bf16 hi (and lo) planes, written as 2 x 16-byte chunks into
// 128B-swizzled tiles (chunks `chunk0`, `chunk0 + 1` of `row`).
template <bool WITH_LO, bool F16 = false>
__device__ __forceinline__ void store_split16(const float* v, uint8_t* tile_hi, uint8_t* tile_lo, int row, int chunk0) {
  uint32_t hi[8], lo[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    hi[i] = pack2<F16>(v[2 * i], v[2 * i + 1]);
    if (WITH_LO) {
      float h0, h1;
      unpack2<F16>(hi[i], h0, h1);
      lo[i] = pack2<F16>(v[2 * i] - h0, v[2 * i + 1] - h1);
    }
  }
  *reinterpret_cast<uint4*>(tile_hi + sw128_offset(row, chunk0)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
  *reinterpret_cast<uint4*>(tile_hi + sw128_offset(row, chunk0 + 1)) = make_uint4(hi[4], hi[5], hi[6], hi[7]);
  if (WITH_LO) {
    *reinterpret_cast<uint4*>(tile_lo + sw128_offset(row, chunk0)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    *reinterpret_cast<uint4*>(tile_lo + sw128_offset(row, chunk0 + 1)) = make_uint4(lo[4], lo[5], lo[6], lo[7]);
  }
}

// 16 fp32 values of one row: bf16 hi packed into 8 TMEM columns (the A operand of a ".ts" MMA), lo (if any) into
// a 128B-swizzled shared-memory tile.
template <bool WITH_LO, bool F16 = false>
__device__ __forceinline__ void store_split16_tmem(const float* v, uint32_t tmem_hi, uint8_t* tile_lo, int row, int chunk0) {
  uint32_t hi[8], lo[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    hi[i] = pack2<F16>(v[2 * i], v[2 * i + 1]);
    if (WITH_LO) {
      float h0, h1;
      unpack2<F16>(hi[i], h0, h1);
      lo[i] = pack2<F16>(v[2 * i] - h0, v[2 * i + 1] - h1);
    }
  }
  tmem_st8(tmem_hi, hi);
  if (WITH_LO) {
    *reinterpret_cast<uint4*>(tile_lo + sw128_offset(row, chunk0)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    *reinterpret_cast<uint4*>(tile_lo + sw128_offset(row, chunk0 + 1)) = make_uint4(lo[4], lo[5], lo[6], lo[7]);
  }
}

// CWG_MODE_F16F8: 16 fp32 values of one row -> fp16 hi / lo tiles (as store_split16<true, true>) plus the two e5m2
// correction planes e5m2((v - hi) * 2^P), e5m2(hi * 2^-Q) as one 16-byte chunk each of [rows x 128 B] tiles.
__device__ __forceinline__ void store_split16_f8(const float* v, uint8_t* tile_hi, uint8_t* tile_lo, uint8_t* tile_l8,
                                                 uint8_t* tile_h8, int row, int chunk0_16, int chunk_8) {
  uint32_t hi[8], lo[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    float h0, h1;
    hi[i] = pack_f16x2(v[2 * i], v[2 * i + 1]);
    unpack2<true>(hi[i], h0, h1);
    lo[i] = pack_f16x2(v[2 * i] - h0, v[2 * i + 1] - h1);
  }
  if (tile_hi) {
    *reinterpret_cast<uint4*>(tile_hi + sw128_offset(row, chunk0_16)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<uint4*>(tile_hi + sw128_offset(row, chunk0_16 + 1)) = make_uint4(hi[4], hi[5], hi[6], hi[7]);
  }
  if (tile_lo) {
    *reinterpret_cast<uint4*>(tile_lo + sw128_offset(row, chunk0_16)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    *reinterpret_cast<uint4*>(tile_lo + sw128_offset(row, chunk0_16 + 1)) = make_uint4(lo[4], lo[5], lo[6], lo[7]);
  }
  uint32_t l8[4], h8[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    l8[i] = e5m2x4_from_f16x2(lo[2 * i], lo[2 * i + 1], F16X2_2P6);
    h8[i] = e5m2x4_from_f16x2(hi[2 * i], hi[2 * i + 1], F16X2_2M8);
  }
  *reinterpret_cast<uint4*>(tile_l8 + sw128_offset(row, chunk_8)) = make_uint4(l8[0], l8[1], l8[2], l8[3]);
  *reinterpret_cast<uint4*>(tile_h8 + sw128_offset(row, chunk_8)) = make_uint4(h8[0], h8[1], h8[2], h8[3]);
}

// CWG_MODE_F16F8 gate output: fp16 hi packed into 8 TMEM columns (A operand of the fp16 ".ts" MMAs) and the two e5m2
// correction planes as one 16-byte chunk each of [rows x 128 B] shared-memory tiles.
__device__ __forceinline__ void store_split16_tmem_f8(const float* v, uint32_t tmem_hi, uint8_t* tile_l8, uint8_t* tile_h8,
                                                      int row, int chunk_8) {
  uint32_t hi[8], lo[8], l8[4], h8[4];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    float h0, h1;
    hi[i] = pack_f16x2(v[2 * i], v[2 * i + 1]);
    unpack2<true>(hi[i], h0, h1);
    lo[i] = pack_f16x2(v[2 * i] - h0, v[2 * i + 1] - h1);
  }
  tmem_st8(tmem_hi, hi);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    l8[i] = e5m2x4_from_f16x2(lo[2 * i], lo[2 * i + 1], F16X2_2P6);
    h8[i] = e5m2x4_from_f16x2(hi[2 * i], hi[2 * i + 1], F16X2_2M8);
  }
  *reinterpret_cast<uint4*>(tile_l8 + sw128_offset(row, chunk_8)) = make_uint4(l8[0], l8[1], l8[2], l8[3]);
  *reinterpret_cast<uint4*>(tile_h8 + sw128_offset(row, chunk_8)) = make_uint4(h8[0], h8[1], h8[2], h8[3]);
}

// tanh(a) * sigmoid(b), glow.py:34-41
template <int NPASS>
__device__ __forceinline__ float gate(float a, float b) {
  if (NPASS != 1) {
    // (1-u)/((1+u)(1+v)), u = e^-2a, v = e^-b : 2 ex2 + 1 rcp, ~1e-6 relative.  Raw .ftz MUFU forms: __expf /
    // __fdividef wrap each MUFU in range-scaling FSETP / predicated FMUL pairs that only matter below 2^-126.
    // a <= -15 saturates (tanh = -1 to 1e-13); v = inf (b < -88) gives 1/inf = 0, the correct limit.
    a = fmaxf(a, -15.f);
    float u, v, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(u) : "f"(a * -2.8853900817779268f));   // -2 * log2(e)
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(v) : "f"(b * -1.4426950408889634f));   // -log2(e)
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"((1.f + u) * (1.f + v)));
    return (1.f - u) * r;
  } else {
    float t, s;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(a));
    asm("tanh.approx.f32 %0, %1;" : "=f"(s) : "f"(0.5f * b));
    return t * fmaf(s, 0.5f, 0.5f);
  }
}

// The same with the bias add folded into the argument scaling: pa, pb are raw accumulator values, ba / bb the biases
// pre-multiplied by GATE_KA / GATE_KB (done once when the biases are staged in shared memory).
template <int NPASS> struct GateK {
  static constexpr float KA = NPASS != 1 ? -2.8853900817779268f : 1.f;     // -2 log2(e) | tanh.approx argument
  static constexpr float KB = NPASS != 1 ? -1.4426950408889634f : 0.5f;    // -log2(e)   | sigmoid(b) = .5 + .5 tanh(b/2)
};
template <int NPASS>
__device__ __forceinline__ float gate_fused(float pa, float pb, float ba, float bb) {
  const float ea = fmaf(pa, GateK<NPASS>::KA, ba), eb = fmaf(pb, GateK<NPASS>::KB, bb);
  if (NPASS != 1) {
    float u, v, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(u) : "f"(fminf(ea, 43.280851f)));   // a >= -15
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(v) : "f"(eb));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"((1.f + u) * (1.f + v)));
    return (1.f - u) * r;
  } else {
    float t, s;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(ea));
    asm("tanh.approx.f32 %0, %1;" : "=f"(s) : "f"(eb));
    return t * fmaf(s, 0.5f, 0.5f);
  }
}

__device__ __forceinline__ void ring_advance(int& slot, uint32_t& phase, int n) {
  if (++slot == n) { slot = 0; phase ^= 1u; }
}

// UMMA descriptor with the address-independent bits precomputed; k-steps add 32 bytes (>>4 = 2).
constexpr uint64_t DESC_SW128_HI = ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
__device__ __forceinline__ void issue_kblock_fast(uint32_t a_addr, uint32_t b_addr, uint32_t tmem_d, uint32_t idesc, bool first) {
  const uint64_t da = DESC_SW128_HI | (uint64_t)((a_addr & 0x3FFFF) >> 4);
  const uint64_t db = DESC_SW128_HI | (uint64_t)((b_addr & 0x3FFFF) >> 4);
  umma_bf16(tmem_d, da, db, idesc, first ? 0u : 1u);
  umma_bf16(tmem_d, da + 2, db + 2, idesc, 1u);
  umma_bf16(tmem_d, da + 4, db + 4, idesc, 1u);
  umma_bf16(tmem_d, da + 6, db + 6, idesc, 1u);
}

// 2 x 16 TMEM columns, issued without waiting; pair with tmem_wait32.
__device__ __forceinline__ void tmem_issue16x2(uint32_t ta, uint32_t tb, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%32];\n\t"
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%33];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(ta), "r"(tb)
      : "memory");
}
__device__ __forceinline__ void tmem_issue16(uint32_t ta, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(ta)
      : "memory");
}
// tcgen05.wait::ld with the destination registers threaded through the asm ("+r"), so that no
// use of them can be scheduled above the wait.
__device__ __forceinline__ void tmem_wait32(uint32_t* r) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]),
                 "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]),
                 "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
               :: "memory");
}
__device__ __forceinline__ void tmem_wait16(uint32_t* r) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
               :: "memory");
}

template <typename K>
inline int set_smem(K kernel, int bytes) {
  CWG_CHECK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  return 0;
}

}}  // namespace cwg::tc
