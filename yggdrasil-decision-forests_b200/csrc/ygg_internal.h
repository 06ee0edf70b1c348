// ygg_internal.h — declarations shared by the translation units of libygg_b200.so (not part of the ABI).
#pragma once
#include <cstdint>
#include <vector>

// Records `msg` as this thread's ygg_last_error() and returns `code`.
__attribute__((visibility("hidden"))) int ygg_set_error_msg(int code, const char* msg);

// Device-resident bucketised dataset (include/ygg_b200.h): bins[f][n_pad] uint8, column-major.
struct ygg_dataset {
  int device = 0;
  int64_t n = 0, n_pad = 0;
  int F = 0;
  uint8_t* d_bins = nullptr;
  int32_t* d_num_bins = nullptr;
  int32_t* d_na_bin = nullptr;
  int32_t* d_feature_type = nullptr;
  float* d_bucket_values = nullptr;   // [F][256] exact threshold rule (ygg_dataset_set_bucket_values), allocated on first use
  int32_t* d_exact_rule = nullptr;    // [F]
  float* d_na_replacement = nullptr;  // [F] NumericalSpec.mean of the features under the exact rule
  std::vector<int32_t> num_bins, na_bin, feature_type;
  int num_sms = 0;
};

__attribute__((visibility("hidden"))) int ygg_internal_dataset_alloc(ygg_dataset** out, int64_t n_rows,
                                                                     int32_t n_features, int32_t device);
__attribute__((visibility("hidden"))) int ygg_internal_dataset_finalize(ygg_dataset* ds);
