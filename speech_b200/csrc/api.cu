// Library introspection entry points of the C ABI (include/speech_b200.h).
#include "common.cuh"

#include "../../include/speech_b200.h"

extern "C" int sb_version(void) { return 101; }

extern "C" const char* sb_status_string(int status) {
  switch (status) {
    case SB_OK: return "ok";
    case SB_ERR_INVALID: return "invalid argument";
    case SB_ERR_CUDA: return "CUDA call failed";
    case SB_ERR_UNSUPPORTED: return "unsupported shape";
    case SB_ERR_WORKSPACE: return "workspace too small";
    default: return "unknown status";
  }
}

extern "C" int sb_device_info(int* sm_count, int* cc_major, int* cc_minor, size_t* l2_bytes) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return SB_ERR_CUDA;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess) return SB_ERR_CUDA;
  if (sm_count) *sm_count = prop.multiProcessorCount;
  if (cc_major) *cc_major = prop.major;
  if (cc_minor) *cc_minor = prop.minor;
  if (l2_bytes) *l2_bytes = (size_t)prop.l2CacheSize;
  return SB_OK;
}

// Levenshtein distance of two int32 token sequences (host code; replaces the `editdistance`
// C extension behind speech/utils/score.py:5,15-16).  Two-row dynamic programme, O(na*nb).
extern "C" long long sb_edit_distance(const int* a, long long na, const int* b, long long nb) {
  if (na < 0 || nb < 0 || (na > 0 && !a) || (nb > 0 && !b)) return -1;
  if (na == 0) return nb;
  if (nb == 0) return na;
  if (nb > na) {   // keep the rows short
    const int* t = a; a = b; b = t;
    const long long tn = na; na = nb; nb = tn;
  }
  long long* row = new long long[nb + 1];
  for (long long j = 0; j <= nb; ++j) row[j] = j;
  for (long long i = 1; i <= na; ++i) {
    long long diag = row[0];
    row[0] = i;
    for (long long j = 1; j <= nb; ++j) {
      const long long up = row[j];
      long long best = diag + (a[i - 1] != b[j - 1] ? 1 : 0);
      if (up + 1 < best) best = up + 1;
      if (row[j - 1] + 1 < best) best = row[j - 1] + 1;
      diag = up;
      row[j] = best;
    }
  }
  const long long d = row[nb];
  delete[] row;
  return d;
}
