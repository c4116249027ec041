// Host-side pieces shared by the tcgen05 engines (sm_100a): the TMA tensor-map encoders and the common shape gate.
// (The first-generation single-CTA kernels that used to live here were retired in round 2: every shape of the path
// is covered by conv_tc2.cu / conv_tc3.cu / conv_tc4.cu; anything else runs on the CUDA-core engine, conv_simt.cu.)
#include <mutex>

#include "tc_common.cuh"

namespace ub {

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(ptr);
  });
  return fn;
}

// 4-D NHWC view {C, W, H, B} with element strides (sw, sh, sb) and a {128 B, TW, TH, 1} box
int encode_act_box(CUtensorMap* m, int dtype, const void* base, int C, int W, int H, int B, long long sw, long long sh,
                   long long sb, int TW, int TH, bool mn_major) {
  EncodeTiledFn enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled entry point not found"); return UNETB200_E_CUDA; }
  const size_t esz = dtype == UNETB200_BF16 ? 2 : 4;
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
  cuuint64_t strides[3] = {(cuuint64_t)(sw * esz), (cuuint64_t)(sh * esz), (cuuint64_t)(sb * esz)};
  cuuint32_t box[4] = {(cuuint32_t)(128 / esz), (cuuint32_t)TW, (cuuint32_t)TH, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(m, dtype == UNETB200_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4,
                   const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   // MN-major fp32 (tf32 wgrad) operands need the 32-byte-atom flavour of the 128-byte swizzle
                   (mn_major && dtype == UNETB200_F32) ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B
                                                       : CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(activation C=%d W=%d H=%d B=%d sw=%lld) failed: %d", C, W, H, B, sw, (int)r);
    return UNETB200_E_CUDA;
  }
  return 0;
}
// bf16 NHWC view {C, W, H, B} with C = 16 / 32 / 64 channels: a {C, box_w, box_h, 1} box whose 2C-byte pixel rows are
// written with the 32 / 64 / 128-byte swizzle (conv_halo.cu)
int encode_act_box_sw(CUtensorMap* m, const void* base, int C, int W, int H, int B, long long sw, long long sh, long long sb,
                      int box_w, int box_h, int esz) {
  EncodeTiledFn enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled entry point not found"); return UNETB200_E_CUDA; }
  if (C != 8 && C != 16 && C != 32 && C != 64) { set_error("encode_act_box_sw: C = %d", C); return UNETB200_E_INVALID; }
  // C = 8: the box is 16 channels wide on an 8-channel tensor -- TMA zero-fills the upper half of every row
  const int box_c = C < 16 ? 16 : C;
  const int row_bytes = box_c * esz;               // 32 / 64 / 128: the swizzle width (bf16: esz 2, fp32 read as TF32: esz 4)
  if ((esz != 2 && esz != 4) || row_bytes > 128) { set_error("encode_act_box_sw: C = %d esz = %d", C, esz); return UNETB200_E_INVALID; }
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
  cuuint64_t strides[3] = {(cuuint64_t)(sw * esz), (cuuint64_t)(sh * esz), (cuuint64_t)(sb * esz)};
  cuuint32_t box[4] = {(cuuint32_t)box_c, (cuuint32_t)box_w, (cuuint32_t)box_h, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(m, esz == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<void*>(base),
                   dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   row_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : (row_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B),
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(narrow activation C=%d W=%d H=%d B=%d sw=%lld) failed: %d", C, W, H, B, sw, (int)r);
    return UNETB200_E_CUDA;
  }
  return 0;
}
int encode_bf16_box(CUtensorMap* m, const void* base, int rank, const unsigned long long* dims, const unsigned long long* strides_bytes,
                    const unsigned* box) {
  EncodeTiledFn enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled entry point not found"); return UNETB200_E_CUDA; }
  if (rank < 2 || rank > 5 || (box[0] != 16 && box[0] != 32 && box[0] != 64)) { set_error("encode_bf16_box: rank %d box %u", rank, box[0]); return UNETB200_E_INVALID; }
  cuuint64_t d[5], st[4];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) { d[i] = dims[i]; bx[i] = box[i]; es[i] = 1; }
  for (int i = 0; i + 1 < rank; ++i) st[i] = strides_bytes[i];
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), d, st, bx, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE,
                   box[0] == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : (box[0] == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B),
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(bf16 box rank %d, inner %u) failed: %d", rank, box[0], (int)r);
    return UNETB200_E_CUDA;
  }
  return 0;
}
int encode_weights(CUtensorMap* m, int dtype, const void* base, int K, int N, int box_n) {
  EncodeTiledFn enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled entry point not found"); return UNETB200_E_CUDA; }
  const size_t esz = dtype == UNETB200_BF16 ? 2 : 4;
  cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)N};
  cuuint64_t strides[1] = {(cuuint64_t)(K * esz)};
  cuuint32_t box[2] = {(cuuint32_t)(128 / esz), (cuuint32_t)box_n};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, dtype == UNETB200_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2,
                   const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(weights K=%d N=%d) failed: %d", K, N, (int)r);
    return UNETB200_E_CUDA;
  }
  return 0;
}

bool tc_common_ok(const unetb200_gconv_t* d) {
  const int esz = d->dtype == UNETB200_BF16 ? 2 : 4;
  const int epr = 128 / esz;
  const int Cq = d->N / d->nquad;
  if (d->Cin % epr || Cq % 64) return false;
  if ((d->ld_in * esz) % 16 || (d->ld_out * esz) % 16) return false;
  if (d->in_scale == 1 && (d->in_off_y || d->in_off_x)) return false;
  if (d->in_scale == 2) {
    if (d->ntaps != 4) return false;
    for (int t = 0; t < 4; ++t)
      if (d->tap_dy[t] != (t >> 1) || d->tap_dx[t] != (t & 1)) return false;
  }
  return true;
}

}  // namespace ub
