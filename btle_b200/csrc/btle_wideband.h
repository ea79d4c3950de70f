// btle_wideband.h — internal interface of the wideband channelizer (btle_wideband.cu).
//
// The C-ABI entry points (btle_b200_wideband_taps / _channelize* / _rx_wideband in btle_rx_kernels.cu) call only
// what is declared here: the tap design and the kernel launch stay inside btle_wideband.cu.
#ifndef BTLE_WIDEBAND_H
#define BTLE_WIDEBAND_H

#include <cuda_runtime.h>

#include <cstddef>
#include <cstdint>
#include <string>
#include <vector>

#include "../../include/btle_b200.h"

namespace btle_wb {

// Checks decim, out_shift and that every channel is 0..39 and inside the band; *err gets the reason.
int validate(const btle_wideband_cfg &cfg, const int32_t *channels, size_t n_ch, std::string *err);

// Complex int16 taps H_q[t] of `channel` (re, im interleaved, 2T values) and the output shift the cfg selects.
int channel_taps(const btle_wideband_cfg &cfg, int channel, std::vector<int16_t> *taps, int *out_shift, std::string *err);

// Number of output samples per channel for n_samples wideband samples: ceil(n_samples / decim).
inline size_t out_samples(size_t n_samples, int decim) { return (n_samples + (size_t)decim - 1) / (size_t)decim; }

// Device state of the channelizer: uploaded taps of the last channel set (reused while it does not change).
struct Scratch {
  void *d_taps = nullptr; size_t taps_bytes = 0;
  cudaEvent_t last_use = nullptr;
  bool used = false, attr_done = false;
  btle_wideband_cfg key_cfg{0, 0, 0, 0};
  std::vector<int32_t> key_channels;
};
void release(Scratch *s);

// Enqueues the channelizer on `st` (arguments already validated; pointers / stride 16-byte aligned).
int launch(Scratch *s, const int8_t *d_wide, size_t n_samples, const btle_wideband_cfg &cfg, const int32_t *channels,
           size_t n_ch, int8_t *d_out, size_t out_stride, cudaStream_t st, std::string *err);

}  // namespace btle_wb

#endif  // BTLE_WIDEBAND_H
