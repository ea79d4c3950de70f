// btle_wideband.cu — exact integer channelizer: one wideband int8 capture (4 MHz x decim) -> 4 Msps int8 captures of
// the BLE channels inside its band, in the receiver's input format (DESIGN.md §6.5).
//
// Contract, per channel (q = channel frequency - centre frequency in MHz, c = (T-1)/2):
//   acc[m] = sum_{t<T} x[m*D + c - t] * H_q[t]            complex int32, x = 0 outside [0, N)
//   rot[m] = acc[m] * (-j)^((q*m) mod 4)                  exact swap / negate of the int32 pair
//   y[m]   = sat8((rot[m] + 2^(s-1)) >> s)                per component; s = 0: no rounding term
// with H_q[t] = round(G * h[t] * exp(+j*2*pi*q*(t-c)/(4D))) from one real, symmetric Kaiser-windowed prototype h.
//
// wideband_kernel: one CTA = kOutTile output samples x kChBlock channels.  The input span of the tile sits in shared
// memory in polyphase order (row = sample index mod D) as words (x[k], x[k+1]) = [I Q I' Q'], so that for a tap pair
// (t, t+1) one 32-bit load feeds both taps of one output, lanes (consecutive outputs) read consecutive words of one
// row, and the tap parity never depends on the output.  The taps of the channel block sit next to it, packed per
// pair as {[Re,-Im]_t, [Im,Re]_t, [Re,-Im]_t+1, [Im,Re]_t+1} (one broadcast 16-byte load).  Per tap pair a thread
// issues kChPerThread 16-byte + kOutPerThread 4-byte shared loads for 4 * kOutPerThread * kChPerThread IDP.2A.
#include "btle_wideband.h"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <mutex>

namespace btle_wb {
namespace {

constexpr int kOutPerThread = 4, kChPerThread = 4;
constexpr int kWarpsOut = 4, kWarpsCh = 2;
constexpr int kThreads = 32 * kWarpsOut * kWarpsCh;
constexpr int kOutTile = 32 * kOutPerThread * kWarpsOut;   // 512 outputs per CTA
constexpr int kChBlock = kChPerThread * kWarpsCh;          // 8 channels per CTA
constexpr size_t kMaxSmem = 232448;

// ---- prototype design ------------------------------------------------------------------------------------------
// Kaiser-windowed sinc, cut-off between the passband edge (0.6 MHz, droop <= 1 dB) and the stopband edge (1.25 MHz,
// >= 50 dB); the shortest odd T whose int16-rounded taps meet both, checked with margins of 0.1 dB / 1 dB.
constexpr double kPassMHz = 0.6, kStopMHz = 1.25, kCutMHz = 0.925;
constexpr double kDesignAttenDb = 53.0, kCheckAttenDb = 51.0, kCheckDroopDb = 0.9;

struct Proto {
  int T = 0, shift = 0;
  std::vector<double> h;         // h[k] = h[c + k] = h[c - k], k = 0..c; sum over all taps = 1
};

double bessel_i0(double x) {
  double s = 1.0, term = 1.0;
  for (int k = 1; k < 200 && term > 1e-17 * s; ++k) { term *= (x / (2.0 * k)) * (x / (2.0 * k)); s += term; }
  return s;
}

// max over f in [f0, f1] of |H(f)| / H(0) for the symmetric taps v[0..c] (v[0] = centre), evaluated on a grid of step df
double response_extreme(const std::vector<double> &v, double fs, double f0, double f1, double df, bool want_min) {
  const int c = (int)v.size() - 1;
  double ref = v[0];
  for (int k = 1; k <= c; ++k) ref += 2.0 * v[k];
  double ext = want_min ? 1e300 : 0.0;
  for (double f = f0; f <= f1 + 1e-12; f += df) {
    const double th = 2.0 * M_PI * f / fs, c1 = cos(th);
    double cm2 = 1.0, cm1 = c1, h = v[0];
    for (int k = 1; k <= c; ++k) {                // cos(k th) by the Chebyshev recurrence
      const double ck = k == 1 ? c1 : 2.0 * c1 * cm1 - cm2;
      if (k > 1) { cm2 = cm1; cm1 = ck; }
      h += 2.0 * v[k] * ck;
    }
    const double a = fabs(h / ref);
    ext = want_min ? std::min(ext, a) : std::max(ext, a);
  }
  return ext;
}

Proto design(int D) {
  const double fs = 4.0 * D, wc = 2.0 * kCutMHz / fs;
  const double beta = 0.1102 * (kDesignAttenDb - 8.7);
  const double est = (kDesignAttenDb - 7.95) / (2.285 * 2.0 * M_PI * (kStopMHz - kPassMHz) / fs);
  int T = std::max(9, ((int)(0.8 * est)) | 1);
  for (;; T += 2) {
    const int c = (T - 1) / 2;
    Proto p;
    p.T = T;
    p.h.resize(c + 1);
    double sum = 0.0, abs_sum = 0.0;
    for (int k = 0; k <= c; ++k) {
      const double r = (double)k / c;
      const double sinc = k == 0 ? wc : sin(M_PI * wc * k) / (M_PI * k);
      p.h[k] = sinc * bessel_i0(beta * sqrt(std::max(0.0, 1.0 - r * r))) / bessel_i0(beta);
      sum += (k ? 2.0 : 1.0) * p.h[k];
    }
    for (double &x : p.h) { x /= sum; }
    for (int k = 0; k <= c; ++k) abs_sum += (k ? 2.0 : 1.0) * fabs(p.h[k]);
    // largest power-of-two gain whose centre tap fits int16 and whose worst rotated accumulator fits int32:
    // |Re| + |Im| <= sqrt(2) |G h| + 1 per tap, 128 * sum < 2^31
    int s = (int)floor(log2(32767.0 / p.h[0]));
    while (s > 0 && 128.0 * (sqrt(2.0) * ldexp(abs_sum, s) + T) >= 2147483648.0) --s;
    p.shift = s;
    std::vector<double> r16(c + 1);
    for (int k = 0; k <= c; ++k) r16[k] = (double)lround(ldexp(p.h[k], s));
    const double df = std::min(0.01, fs / (16.0 * T));
    const double pass = response_extreme(r16, fs, 0.0, kPassMHz, 0.01, true);
    const double stop = response_extreme(r16, fs, kStopMHz, fs / 2.0, df, false);
    if (20.0 * log10(pass) >= -kCheckDroopDb && 20.0 * log10(stop) <= -kCheckAttenDb) return p;
  }
}

const Proto &proto(int D) {
  static std::mutex mu;
  static Proto cache[65];
  std::lock_guard<std::mutex> lock(mu);
  if (!cache[D].T) cache[D] = design(D);
  return cache[D];
}

int freq_mhz(int ch) { return (int)(btle_b200_get_freq_by_channel_number(ch) / 1000000ull); }

// ---- kernel ------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads, 2)
wideband_kernel(const uint16_t *__restrict__ x, long long n_samples, long long n_out, const uint4 *__restrict__ taps,
                const int *__restrict__ qch, int n_pairs, int c, int D, int L, int qmin, int n_ch, int n_cb,
                int8_t *__restrict__ out, long long stride, int shift) {
  extern __shared__ uint4 smem[];
  uint4 *s_taps = smem;                                                   // [kChBlock][n_pairs]
  int *s_off = reinterpret_cast<int *>(s_taps + kChBlock * n_pairs);      // [n_pairs], padded to 16 bytes
  uint32_t *s_tile = reinterpret_cast<uint32_t *>(s_off + ((n_pairs + 3) & ~3));   // [D][L]
  const int cb = (int)(blockIdx.x % (unsigned)n_cb);
  const long long m0 = (long long)(blockIdx.x / (unsigned)n_cb) * kOutTile;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  const uint4 *g_taps = taps + (size_t)cb * kChBlock * n_pairs;
  for (int i = tid; i < kChBlock * n_pairs; i += kThreads) s_taps[i] = g_taps[i];
  for (int p = tid; p < n_pairs; p += kThreads) {
    const int e = c - 2 * p - 1;                                          // word (x[k-1], x[k]) of tap pair p: k-1 = m*D + e
    const int q = e >= 0 ? e / D : -((-e + D - 1) / D);
    s_off[p] = (e - q * D) * L + (q - qmin);
  }
  const long long kb = (m0 + qmin) * D;                                   // tile column j, row r <-> sample kb + j*D + r
  for (int i = tid; i < D * L; i += kThreads) {
    const long long g = kb + i;
    const uint32_t lo = (g >= 0 && g < n_samples) ? x[g] : 0u;
    const uint32_t hi = (g + 1 >= 0 && g + 1 < n_samples) ? x[g + 1] : 0u;
    const int j = i / D;
    s_tile[(i - j * D) * L + j] = lo | (hi << 16);
  }
  __syncthreads();

  const int ob = (warp % kWarpsOut) * 32 * kOutPerThread + lane;          // local output of r = 0
  const int cl = (warp / kWarpsOut) * kChPerThread;                       // first local channel
  int acc_re[kOutPerThread][kChPerThread], acc_im[kOutPerThread][kChPerThread];
#pragma unroll
  for (int r = 0; r < kOutPerThread; ++r)
#pragma unroll
    for (int j = 0; j < kChPerThread; ++j) acc_re[r][j] = acc_im[r][j] = 0;

#pragma unroll 2
  for (int p = 0; p < n_pairs; ++p) {
    const int off = s_off[p] + ob;
    uint4 tp[kChPerThread];
#pragma unroll
    for (int j = 0; j < kChPerThread; ++j) tp[j] = s_taps[(cl + j) * n_pairs + p];
#pragma unroll
    for (int r = 0; r < kOutPerThread; ++r) {
      const int w = (int)s_tile[off + 32 * r];                            // bytes [I Q] of x[k-1], then of x[k]
#pragma unroll
      for (int j = 0; j < kChPerThread; ++j) {
        acc_re[r][j] = __dp2a_hi((int)tp[j].x, w, acc_re[r][j]);           // tap t   x x[k]
        acc_im[r][j] = __dp2a_hi((int)tp[j].y, w, acc_im[r][j]);
        acc_re[r][j] = __dp2a_lo((int)tp[j].z, w, acc_re[r][j]);           // tap t+1 x x[k-1]
        acc_im[r][j] = __dp2a_lo((int)tp[j].w, w, acc_im[r][j]);
      }
    }
  }

  const long long round_add = shift ? (1ll << (shift - 1)) : 0ll;
#pragma unroll
  for (int j = 0; j < kChPerThread; ++j) {
    const int ch = cb * kChBlock + cl + j;
    const int q = qch[cb * kChBlock + cl + j];
#pragma unroll
    for (int r = 0; r < kOutPerThread; ++r) {
      const long long m = m0 + ob + 32 * r;
      const long long a = acc_re[r][j], b = acc_im[r][j];
      const int rot = (int)(((long long)q * m) & 3);                      // (-j)^rot
      const long long re = rot == 0 ? a : rot == 1 ? b : rot == 2 ? -a : -b;
      const long long im = rot == 0 ? b : rot == 1 ? -a : rot == 2 ? -b : a;
      const int yr = (int)max(-128ll, min(127ll, (re + round_add) >> shift));
      const int yi = (int)max(-128ll, min(127ll, (im + round_add) >> shift));
      if (ch < n_ch && m < n_out)
        *reinterpret_cast<uint16_t *>(out + ch * stride + 2 * m) = (uint16_t)((yr & 0xFF) | ((yi & 0xFF) << 8));
    }
  }
}

uint32_t pack16(int lo, int hi) { return (uint32_t)(uint16_t)(int16_t)lo | ((uint32_t)(uint16_t)(int16_t)hi << 16); }

}  // namespace

int validate(const btle_wideband_cfg &cfg, const int32_t *channels, size_t n_ch, std::string *err) {
  if (cfg.decim < 2 || cfg.decim > 64) { *err = "wideband decim must be 2..64 (sample rate 8..256 Msps)"; return BTLE_EINVAL; }
  if (cfg.out_shift < -1 || cfg.out_shift > 31) { *err = "wideband out_shift must be -1 (default) or 0..31"; return BTLE_EINVAL; }
  if (n_ch && !channels) { *err = "channel list is NULL"; return BTLE_EINVAL; }
  for (size_t i = 0; i < n_ch; ++i) {
    if (channels[i] < 0 || channels[i] > 39) { *err = "channel number must be within 0~39"; return BTLE_EINVAL; }
    const int q = freq_mhz(channels[i]) - cfg.center_mhz;
    if (std::abs(q) + 1 > 2 * cfg.decim) {
      *err = "channel " + std::to_string(channels[i]) + " (" + std::to_string(freq_mhz(channels[i])) + " MHz) is outside the band of " +
             std::to_string(4 * cfg.decim) + " Msps around " + std::to_string(cfg.center_mhz) + " MHz";
      return BTLE_EINVAL;
    }
  }
  return BTLE_OK;
}

int channel_taps(const btle_wideband_cfg &cfg, int channel, std::vector<int16_t> *taps, int *out_shift, std::string *err) {
  int rc = validate(cfg, &channel, 1, err);
  if (rc) return rc;
  const Proto &p = proto(cfg.decim);
  const int T = p.T, c = (T - 1) / 2, period = 4 * cfg.decim;
  const int q = freq_mhz(channel) - cfg.center_mhz;
  const double G = ldexp(1.0, p.shift);
  taps->resize(2 * (size_t)T);
  double bound = 0.0;
  for (int t = 0; t < T; ++t) {
    const int a = (int)((((long long)q * (t - c)) % period + period) % period);   // exp(+j 2 pi q (t-c) / (4D)), exact angle
    const double g = G * p.h[std::abs(t - c)], ang = 2.0 * M_PI * a / period;
    const long re = std::min(32767l, std::max(-32767l, lround(g * cos(ang))));
    const long im = std::min(32767l, std::max(-32767l, lround(g * sin(ang))));
    (*taps)[2 * t] = (int16_t)re;
    (*taps)[2 * t + 1] = (int16_t)im;
    bound += (double)(std::abs(re) + std::abs(im));
  }
  if (128.0 * bound >= 2147483648.0) { *err = "internal: channel taps could overflow int32"; return BTLE_EINVAL; }
  *out_shift = cfg.out_shift >= 0 ? cfg.out_shift : p.shift;
  return BTLE_OK;
}

void release(Scratch *s) {
  if (s->d_taps) cudaFree(s->d_taps);
  if (s->last_use) cudaEventDestroy(s->last_use);
  *s = Scratch();
}

int launch(Scratch *s, const int8_t *d_wide, size_t n_samples, const btle_wideband_cfg &cfg, const int32_t *channels,
           size_t n_ch, int8_t *d_out, size_t out_stride, cudaStream_t st, std::string *err) {
  if (!n_ch || !n_samples) return BTLE_OK;
  const int D = cfg.decim;
  const Proto &p = proto(D);
  const int T = p.T, c = (T - 1) / 2, n_pairs = (T + 1) / 2;
  const int n_cb = (int)((n_ch + kChBlock - 1) / kChBlock), n_chp = n_cb * kChBlock;
  const size_t taps_bytes = (size_t)n_chp * n_pairs * sizeof(uint4), bytes = taps_bytes + (size_t)n_chp * sizeof(int);
  const bool same = s->d_taps && s->key_cfg.decim == cfg.decim && s->key_cfg.center_mhz == cfg.center_mhz &&
                    s->key_cfg.out_shift == cfg.out_shift && s->key_channels.size() == n_ch &&
                    std::equal(channels, channels + n_ch, s->key_channels.begin());
  if (!same) {
    if (!s->last_use && cudaEventCreateWithFlags(&s->last_use, cudaEventDisableTiming) != cudaSuccess) {
      cudaGetLastError(); *err = "cudaEventCreate failed"; return BTLE_ECUDA;
    }
    if (s->taps_bytes < bytes) {
      if (s->d_taps) cudaFree(s->d_taps);                                 // (waits for launches still reading it)
      s->d_taps = nullptr; s->taps_bytes = 0; s->used = false;
      if (cudaMalloc(&s->d_taps, bytes) != cudaSuccess) { cudaGetLastError(); *err = "cudaMalloc failed"; return BTLE_ENOMEM; }
      s->taps_bytes = bytes;
    }
    std::vector<uint4> packed((size_t)n_chp * n_pairs, uint4{0, 0, 0, 0});
    std::vector<int> qs(n_chp, 0);
    std::vector<int16_t> h;
    int shift = 0;
    for (size_t i = 0; i < n_ch; ++i) {
      const int rc = channel_taps(cfg, channels[i], &h, &shift, err);
      if (rc) return rc;
      qs[i] = freq_mhz(channels[i]) - cfg.center_mhz;
      h.resize(2 * (size_t)(T + 1), 0);                                   // tap T = 0: pairs cover T + 1 taps
      for (int pr = 0; pr < n_pairs; ++pr) {
        const int r0 = h[4 * pr], i0 = h[4 * pr + 1], r1 = h[4 * pr + 2], i1 = h[4 * pr + 3];
        packed[i * n_pairs + pr] = uint4{pack16(r0, -i0), pack16(i0, r0), pack16(r1, -i1), pack16(i1, r1)};
      }
    }
    // a launch on another stream may still read the previous taps
    if (s->used && cudaStreamWaitEvent(st, s->last_use, 0) != cudaSuccess) { cudaGetLastError(); *err = "cudaStreamWaitEvent failed"; return BTLE_ECUDA; }
    if (cudaMemcpyAsync(s->d_taps, packed.data(), taps_bytes, cudaMemcpyHostToDevice, st) != cudaSuccess ||
        cudaMemcpyAsync(static_cast<char *>(s->d_taps) + taps_bytes, qs.data(), n_chp * sizeof(int), cudaMemcpyHostToDevice, st) != cudaSuccess ||
        cudaStreamSynchronize(st) != cudaSuccess) {                       // host staging vectors die at return
      cudaGetLastError(); *err = "tap upload failed"; return BTLE_ECUDA;
    }
    s->key_cfg = cfg;
    s->key_channels.assign(channels, channels + n_ch);
  }
  const int qmin = -((c + 1 + D - 1) / D);                                // floor((-c-1) / D)
  const int qmax = (c - 1) >= 0 ? (c - 1) / D : -1;
  int L = kOutTile + qmax - qmin;
  L |= 1;                                                                 // odd row pitch: the strided tile fill is bank-conflict free
  const size_t smem = (size_t)kChBlock * n_pairs * sizeof(uint4) + (size_t)((n_pairs + 3) & ~3) * sizeof(int) + (size_t)D * L * sizeof(uint32_t);
  if (smem > kMaxSmem) { *err = "internal: channelizer tile exceeds shared memory"; return BTLE_EINVAL; }
  if (!s->attr_done) {
    if (cudaFuncSetAttribute(wideband_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem) != cudaSuccess) {
      cudaGetLastError(); *err = "cudaFuncSetAttribute failed"; return BTLE_ECUDA;
    }
    s->attr_done = true;
  }
  const long long n_out = (long long)out_samples(n_samples, D);
  const long long tiles = (n_out + kOutTile - 1) / kOutTile;
  if (tiles * n_cb > 0x7FFFFFFFll) { *err = "wideband capture too large for one launch"; return BTLE_EINVAL; }
  wideband_kernel<<<(unsigned)(tiles * n_cb), kThreads, smem, st>>>(
      reinterpret_cast<const uint16_t *>(d_wide), (long long)n_samples, n_out, static_cast<const uint4 *>(s->d_taps),
      reinterpret_cast<const int *>(static_cast<const char *>(s->d_taps) + taps_bytes), n_pairs, c, D, L, qmin, (int)n_ch, n_cb, d_out,
      (long long)out_stride, cfg.out_shift >= 0 ? cfg.out_shift : p.shift);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaEventRecord(s->last_use, st);
  if (e != cudaSuccess) { *err = std::string("wideband_kernel: ") + cudaGetErrorString(e); return BTLE_ECUDA; }
  s->used = true;
  return BTLE_OK;
}

}  // namespace btle_wb
