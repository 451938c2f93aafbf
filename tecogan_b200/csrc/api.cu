// Error plumbing and device queries for the C ABI (include/teco.h).
#include <stdarg.h>
#include <string.h>
#include "teco_common.cuh"

static thread_local char g_err[512] = "";

void teco_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int teco_sm_count() {
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (sms <= 0) sms = 148;
  }
  return sms;
}

int teco_tmap_bf16(CUtensorMap* map, const char* who, const void* base, int rank, const cuuint64_t* dims, const cuuint64_t* strides,
                   const cuuint32_t* box) {
  typedef CUresult (*EncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static EncodeTiled enc = nullptr;
  if (!enc) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      enc = (EncodeTiled)p;
  }
  if (!enc) {
    teco_set_error("%s: cuTensorMapEncodeTiled is unavailable (no CUDA driver?)", who);
    return TECO_E_CUDA;
  }
  const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  const CUresult cr = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (cr != CUDA_SUCCESS) {
    teco_set_error("%s: cuTensorMapEncodeTiled failed with CUresult %d (rank %d, innermost dimensions %llu x %llu)", who, (int)cr, rank,
                   (unsigned long long)dims[0], (unsigned long long)dims[1]);
    return TECO_E_CUDA;
  }
  return TECO_OK;
}

int teco_tmap_nhwc(CUtensorMap* map, const char* who, const void* base, int N, int H, int W, int C, int box_c, int box_w, int box_h) {
  const cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  const cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  const cuuint32_t box[4] = {(cuuint32_t)box_c, (cuuint32_t)box_w, (cuuint32_t)box_h, 1};
  return teco_tmap_bf16(map, who, base, 4, dims, strides, box);
}

extern "C" {

const char* teco_last_error(void) { return g_err; }

int teco_version(void) { return 100; }

int teco_device_props(int device, int64_t* props) {
  TECO_CHECK_ARG(props != nullptr, "teco_device_props: props is NULL");
  cudaDeviceProp p;
  TECO_CUDA_CALL(cudaGetDeviceProperties(&p, device));
  props[0] = p.multiProcessorCount;
  props[1] = p.major;
  props[2] = p.minor;
  props[3] = (int64_t)p.sharedMemPerBlockOptin;
  props[4] = (int64_t)p.l2CacheSize;
  props[5] = props[6] = props[7] = 0;
  return TECO_OK;
}

// CRC32C (Castagnoli, reflected 0x82F63B78), slicing-by-8 on the host: checkpoint files (tecogan_b200/tf_bundle.py)
// carry a masked CRC32C per table block and per tensor; this is host-side utility code, no device work.
int64_t teco_crc32c(const void* data, int64_t n, int64_t crc_in) {
  if ((!data && n > 0) || n < 0 || crc_in < 0 || crc_in > 0xFFFFFFFFll) {
    teco_set_error("teco_crc32c: bad argument");
    return TECO_E_INVALID;
  }
  static uint32_t tab[8][256];
  static bool init = false;
  if (!init) {
    for (uint32_t i = 0; i < 256; ++i) {
      uint32_t c = i;
      for (int k = 0; k < 8; ++k) c = (c & 1) ? (c >> 1) ^ 0x82F63B78u : c >> 1;
      tab[0][i] = c;
    }
    for (uint32_t i = 0; i < 256; ++i)
      for (int t = 1; t < 8; ++t) tab[t][i] = (tab[t - 1][i] >> 8) ^ tab[0][tab[t - 1][i] & 0xFF];
    init = true;
  }
  const uint8_t* p = (const uint8_t*)data;
  uint32_t c = (uint32_t)crc_in ^ 0xFFFFFFFFu;
  while (n >= 8) {
    uint32_t lo, hi;
    memcpy(&lo, p, 4);
    memcpy(&hi, p + 4, 4);
    lo ^= c;
    c = tab[7][lo & 0xFF] ^ tab[6][(lo >> 8) & 0xFF] ^ tab[5][(lo >> 16) & 0xFF] ^ tab[4][lo >> 24] ^ tab[3][hi & 0xFF] ^
        tab[2][(hi >> 8) & 0xFF] ^ tab[1][(hi >> 16) & 0xFF] ^ tab[0][hi >> 24];
    p += 8;
    n -= 8;
  }
  while (n-- > 0) c = tab[0][(c ^ *p++) & 0xFF] ^ (c >> 8);
  return (int64_t)(c ^ 0xFFFFFFFFu);
}

}  // extern "C"
