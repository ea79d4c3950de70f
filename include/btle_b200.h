/* btle_b200 — C-ABI of the Blackwell-native BLE receive baseband.
 *
 * Drop-in boundary for ONE path of JiaoXianjun/BTLE: the btle_rx receive chain
 *   int8 IQ @4 Msps -> GFSK differential demod -> 4:1 bit decision -> 32-bit masked
 *   access-address sliding match -> dewhiten -> header parse -> CRC-24
 * (reference: host/btle-tools/src/btle_rx.c:1489-1562, 1969-2016, 2188-2391).
 *
 * The reference has no library/FFI layer (btle_rx is one translation unit,
 * src/CMakeLists.txt:34); its only function seam for this path is
 *   void receiver(IQ_TYPE *rxp_in, int buf_len, int channel_number, uint32_t access_addr,
 *                 uint32_t crc_init, int verbose_flag, int raw_flag)        btle_rx.c:2188
 * called by main() once per 16384-int8 half of its ring buffer (btle_rx.c:2619-2651), with the
 * mask, filters and sinks passed through globals.  btle_b200_rx*() replaces that call for a
 * whole capture (or a batch of captures) at once and RETURNS the packets receiver() would
 * have counted, in the same order, instead of printing them.  See INTEGRATION.md for the
 * binding a maintainer of the reference would add.
 *
 * Plain C: pointers and sizes only.  Every function returns 0 or a negative BTLE_E* code and
 * never exits the process.  A context is bound to one CUDA device and is not thread-safe;
 * use one context per thread.  There is NO CPU fallback: without a CUDA device
 * btle_b200_create() fails with BTLE_ENODEV.
 */
#ifndef BTLE_B200_H
#define BTLE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BTLE_OK 0
#define BTLE_EINVAL (-1)   /* bad argument (channel > 39, misaligned device pointer, ...)   */
#define BTLE_ENODEV (-2)   /* no usable CUDA device                                          */
#define BTLE_ENOMEM (-3)   /* device or host allocation failed                               */
#define BTLE_ECUDA (-4)    /* a CUDA call failed; see btle_b200_last_error()                 */
#define BTLE_EOVERFLOW (-5)/* more packets than `cap`; *n_out holds the number found          */
/* btle_b200_search_unique_bits() returns sample indices (even values >= -248, or -1 = no match, like the
 * reference's function), so its errors are moved out of that range: BTLE_SEARCH_ERR(BTLE_ECUDA) == -1004. */
#define BTLE_SEARCH_ERR(code) ((code) - 1000)

#define BTLE_CHUNK_INT8 16384      /* LEN_BUF/2, btle_rx.c:223-224                           */
#define BTLE_LOOKAHEAD_INT8 3008   /* LEN_BUF_MAX_NUM_PHY_SAMPLE, btle_rx.c:237-238          */
/* Upper bound of packets receiver() can count in one chunk.  A packet moves buf_len_eaten on by at least
 * 2*n0' + 256 + 64*2 + 64*3 int8 (:2226-2232, :2259, :2305) where n0' >= -4*ctz(access_addr & mask) relative to
 * the restart point (zeroed history, :1518), and a new search starts only while buf_len_eaten < 16632 (:2218):
 * 34 per chunk when bit 0 of the masked access address is set, 51 in the degenerate case mask == 0.  Real
 * captures hold a few; callers may size `cap` smaller and grow it on BTLE_EOVERFLOW (*n_out = needed). */
#define BTLE_MAX_PKTS_PER_CHUNK 51

/* Per-capture receiver parameters == btle_rx's -c / -a / -m / -k / -r / -R options
 * (parse_commandline, btle_rx.c:1244-1458; defaults :1271-1301). */
typedef struct {
  int32_t channel;       /* -c  0..39; 37..39 select the advertising-PDU header parser       */
  uint32_t access_addr;  /* -a  default 0x8E89BED6                                           */
  uint32_t access_mask;  /* -m  default 0xFFFFFFFF; bit p = compare p-th received AA bit     */
  uint32_t crc_init;     /* -k  default 0x555555, NOT reordered (crc_init_reorder is ours)   */
  int32_t raw;           /* -r  1: 42 un-dewhitened bytes after each AA hit (btle_rx.c:2254) */
  int32_t rssi;          /* flag bits: BTLE_CFG_RSSI (-R) 1: also return sum|I|+|Q| over the AA samples
                            (:2234-2243); BTLE_CFG_REPORT_REJECTED (-v) 2: advertising-channel hits whose header
                            length is outside 6..37 — the reference prints "PktBAD" for them under -v and does not
                            count them (:2291-2298) — come back as records with BTLE_REC_REJECTED set (at most 16
                            per chunk)                                                                           */
} btle_stream_cfg;
#define BTLE_CFG_RSSI 1
#define BTLE_CFG_REPORT_REJECTED 2

/* One packet the reference would have counted (pkt_count++, btle_rx.c:2274/:2319). 64 bytes. */
typedef struct {
  int32_t stream;        /* index of the capture in the batch                                */
  int32_t chunk;         /* index of the 16384-int8 chunk receiver() would have been given    */
  int32_t n0;            /* first IQ sample of the access address, relative to that chunk
                            (-124..8191; == hit_idx/2 accumulated, btle_rx.c:2226)            */
  uint8_t channel;
  uint8_t n_bytes;       /* 42 in raw mode, else 2 + payload_len + 3                          */
  uint8_t crc_bad;       /* crc_check() verdict, 1 = mismatch (btle_rx.c:2015); 0 in raw mode */
  uint8_t flags;         /* bit0 raw, bit1 advertising channel, bit2 BTLE_REC_REJECTED: not a packet the
                            reference counts — only bytes[0..1] (the header) are valid, n_bytes = 2      */
  uint32_t access_addr;
  uint16_t mag_sum;      /* sum |I|+|Q| over the 128 AA samples if cfg.rssi, else 0           */
  uint8_t bytes[42];     /* == reference tmp_byte[] (btle_rx.c:1485): dewhitened header,
                            payload, CRC; zero beyond n_bytes                                 */
} btle_pkt_rec;

#define BTLE_REC_REJECTED 4

typedef struct btle_b200_ctx btle_b200_ctx;

/* ---- context -------------------------------------------------------------------------- */
int btle_b200_create(btle_b200_ctx **out, int cuda_device);
void btle_b200_destroy(btle_b200_ctx *ctx);
const char *btle_b200_last_error(const btle_b200_ctx *ctx);
const char *btle_b200_strerror(int code);
/* Host placement for the host-buffer entry points: binds the CALLING THREAD to the CPUs of the NUMA node the GPU's
 * PCIe root hangs off (sysfs numa_node / cpulist, intersected with the current affinity) and makes that node the
 * preferred one for its page allocations.  Call it before allocating (page-locked) IQ buffers: on a two-socket box
 * host->device copies from the far socket cross the inter-socket link and the 8 GPUs' copies then share it.
 * *node_out = the node, or -1 if the machine does not expose one (then nothing is changed). */
int btle_b200_bind_host_numa(int cuda_device, int *node_out);
/* library/ABI version, (major<<16)|minor */
uint32_t btle_b200_version(void);

/* ---- the hot path --------------------------------------------------------------------- */
/* Host buffers in, host records out (what a reference-side caller uses; replaces the
 * main()->receiver() loop, btle_rx.c:2610-2662).  `iq` holds n_streams captures; capture s
 * starts at iq + s*stream_stride_int8 and is n_int8 long (interleaved I,Q int8, as written
 * by rx_callback, btle_rx.c:531-540).  Chunk k of a capture exists while 16384(k+1) <= n_int8;
 * bytes past the end of a capture read as 0 (the reference would wait for the radio).
 * Records come back sorted by (stream, chunk, n0) == the order receiver() emits them.
 * `iq` may be page-locked (cudaHostAlloc / cudaHostRegister: copied by DMA directly) or ordinary pageable
 * memory (moved through the context's page-locked staging buffers in 32 MiB segments, CPU copy of one
 * segment overlapping the DMA of the previous one). */
int btle_b200_rx_batch(btle_b200_ctx *ctx, const int8_t *iq, size_t n_streams, size_t stream_stride_int8,
                       size_t n_int8, const btle_stream_cfg *cfgs, btle_pkt_rec *out, size_t cap,
                       size_t *n_out);
/* Single capture convenience wrapper. */
int btle_b200_rx(btle_b200_ctx *ctx, const int8_t *iq, size_t n_int8, const btle_stream_cfg *cfg,
                 btle_pkt_rec *out, size_t cap, size_t *n_out);

/* Device-resident variant: `d_iq` (16-byte aligned; stride a multiple of 16 when n_streams > 1), `d_out`, `d_count`
 * and `d_dir` are device pointers usable from the context's device (local HBM or PEER memory of another GPU —
 * that is how the multi-GPU gather works: every rank's kernel stores its records straight into rank 0's buffer
 * over NVLink); work is enqueued on `cuda_stream` (a cudaStream_t, may be NULL) and NOT synchronised.
 *
 * Output layout.  A launch is cut into btle_b200_rx_units() UNITS of work (16 chunks of one capture, or a few
 * chunks in the last wave of the persistent grid), numbered in (stream, chunk) order.  Each unit reserves ONE
 * contiguous block of d_out (one atomic per unit on *d_count) and writes its records there in the reference's
 * order, and fills d_dir[unit] = {first record, number of records}.  So:
 *   - walking d_dir in index order visits all records in the order receiver() emits them (no sort needed);
 *     btle_b200_gather_ordered() does that walk on host copies;
 *   - sum(d_dir[u].count) == *d_count == packets found, also when that exceeds `cap` (records beyond cap are
 *     not stored);
 *   - blocks themselves follow each other in the order the units finished, i.e. d_out as a whole is NOT sorted.
 * *d_count (uint32) is zeroed by the call; every d_dir entry of the launch is written (no memset needed).
 * btle_b200_rx_device_dir() accepts d_count == NULL: the block reservations then run on a context-owned counter (a ring
 * of them, each cleared by an earlier launch) and no memset is enqueued in front of the kernel — for callers that take
 * the packet count from the directory. */
typedef struct { uint32_t base, count; } btle_unit_dir;
size_t btle_b200_rx_units(const btle_b200_ctx *ctx, size_t n_streams, size_t n_int8);
int btle_b200_rx_device_dir(btle_b200_ctx *ctx, const int8_t *d_iq, size_t n_streams, size_t stream_stride_int8,
                            size_t n_int8, const btle_stream_cfg *cfgs, btle_pkt_rec *d_out, size_t cap,
                            uint32_t *d_count, btle_unit_dir *d_dir, size_t dir_cap, void *cuda_stream);
/* Same with the directory kept in context-owned scratch: for callers that only want the set of records
 * (btle_b200_sort_records() on the host copy gives reference order). */
int btle_b200_rx_device(btle_b200_ctx *ctx, const int8_t *d_iq, size_t n_streams, size_t stream_stride_int8,
                        size_t n_int8, const btle_stream_cfg *cfgs, btle_pkt_rec *d_out, size_t cap,
                        uint32_t *d_count, void *cuda_stream);
void btle_b200_sort_records(btle_pkt_rec *recs, size_t n);
/* Host helper: recs[0..n_recs) and dir[0..n_units) are host copies of a launch's d_out / d_dir; copies the
 * records into out[] in reference order.  *n_out = sum of the directory counts; BTLE_EOVERFLOW if that exceeds
 * `cap` or if blocks were cut off by n_recs (out then holds what was available, still in order). */
int btle_b200_gather_ordered(const btle_pkt_rec *recs, size_t n_recs, const btle_unit_dir *dir, size_t n_units,
                             btle_pkt_rec *out, size_t cap, size_t *n_out);
/* ---- streaming session: ONE capture of unbounded length (file, pipe, radio), pushed in pieces -------------------
 * The library cuts the stream into segments of `segment_chunks` chunks (0 = default 4096 = 64 MiB) and double-buffers
 * them: while the GPU copies / decodes segment i out of one page-locked buffer, the caller fills the other with
 * segment i+1 (btle_b200_stream_acquire() hands out that buffer directly, so a file can be read() straight into
 * page-locked memory; btle_b200_stream_push() is the copying convenience form).  Capture size is therefore bounded
 * neither by host RAM nor by HBM.  Records come back in the reference's order, `chunk` counted from the start of the
 * stream, as segments complete (the calls return how many they stored; they never block on the segment just handed
 * over).  Chunk semantics are the batch entry points': a chunk exists once its 16384 int8 are there, decode reads up
 * to 3008 int8 behind it, bytes behind the end of the stream read as 0. */
typedef struct btle_b200_stream btle_b200_stream;
int btle_b200_stream_open(btle_b200_ctx *ctx, const btle_stream_cfg *cfg, size_t segment_chunks, btle_b200_stream **out);
int btle_b200_stream_acquire(btle_b200_stream *s, int8_t **buf, size_t *space);       /* where to put the next bytes    */
int btle_b200_stream_commit(btle_b200_stream *s, size_t n_int8, btle_pkt_rec *out, size_t cap, size_t *n_out);
int btle_b200_stream_push(btle_b200_stream *s, const int8_t *iq, size_t n_int8, btle_pkt_rec *out, size_t cap, size_t *n_out);
/* retune: channel / access address / CRC init used from the next segment on (hop following on a live stream) */
int btle_b200_stream_set_cfg(btle_b200_stream *s, const btle_stream_cfg *cfg);
/* end of stream: decodes the tail, returns what is left (BTLE_EOVERFLOW: call again, more records are waiting) */
int btle_b200_stream_finish(btle_b200_stream *s, btle_pkt_rec *out, size_t cap, size_t *n_out);
void btle_b200_stream_close(btle_b200_stream *s);

/* number of kernels the last rx call launched (bench.py's gpu_launches) */
int btle_b200_last_launches(const btle_b200_ctx *ctx);

/* ---- leaf functions with the reference's signatures (unit parity; each runs on the GPU) ---- */
/* search_unique_bits, btle_rx.c:1510: returns the int8 index of the first AA sample of the
 * first match when scanning `search_len` symbols from rxp with a zeroed history, or -1.
 * unique_bits / unique_bits_mask are 32 bytes of 0/1, LSB first (uint32_to_bit_array, :798).
 * Reads rxp[0 .. 8*search_len+1]; search_len <= 4096.  Errors: BTLE_SEARCH_ERR(BTLE_E*) (<= -1001). */
int btle_b200_search_unique_bits(btle_b200_ctx *ctx, const int8_t *rxp, int search_len,
                                 const uint8_t *unique_bits, const uint8_t *unique_bits_mask, int num_bits);
/* demod_byte, btle_rx.c:1489: num_byte <= 64 bytes from rxp[0 .. 64*num_byte+3]. */
int btle_b200_demod_byte(btle_b200_ctx *ctx, const int8_t *rxp, int num_byte, uint8_t *out_byte);
/* scramble_byte with scramble_table[channel]+table_offset, btle_rx.c:1232 / scramble_table.h:4. */
int btle_b200_scramble_byte(btle_b200_ctx *ctx, const uint8_t *byte_in, int num_byte, int channel,
                            int table_offset, uint8_t *byte_out);
/* crc24_byte, btle_rx.c:1224 (init_hex already reordered), and crc_init_reorder, :1969. */
int btle_b200_crc24_byte(btle_b200_ctx *ctx, const uint8_t *byte_in, int num_byte, uint32_t init_hex,
                         uint32_t *crc_out);
uint32_t btle_b200_crc_init_reorder(uint32_t crc_init);
/* parse_adv_pdu_header_byte :1947 / parse_ll_pdu_header_byte :1939 (host-side, pure bit ops). */
void btle_b200_parse_adv_pdu_header_byte(const uint8_t *byte_in, int *pdu_type, int *tx_add, int *rx_add,
                                         int *payload_len);
void btle_b200_parse_ll_pdu_header_byte(const uint8_t *byte_in, int *llid, int *nesn, int *sn, int *md,
                                        int *payload_len);
/* Discriminator bits d[n] = (I[n]Q[n+1]-I[n+1]Q[n]) > 0 for n < n_samples (one byte 0/1 each);
 * reads iq[0 .. 2*n_samples+1] (host pointers). */
int btle_b200_dbits(btle_b200_ctx *ctx, const int8_t *iq, size_t n_samples, uint8_t *d_out);

/* ---- leaf functions with the signatures of the reference's bit-true Python model
 *      (python/btlelib.py; arrays of 0/1 int8 "bits", int16 samples at symbol rate) ------------- */
/* gfsk_demodulation_fixed_point(i, q), btlelib.py:395-400: for k < n-1
 *   signal[k] = int32(i[k])*int32(q[k+1]) - int32(i[k+1])*int32(q[k]),  bit[k] = signal[k] > 0. */
int btle_b200_gfsk_demod_i16(btle_b200_ctx *ctx, const int16_t *i, const int16_t *q, size_t n, int8_t *bit_out,
                             int32_t *signal_out);
/* search_unique_bit_sequence(bit, bit_sequence), btlelib.py:402-412: first index where the
 * sequence occurs, or -1 (also the function's return; errors are <= -2... see BTLE_E*). */
long btle_b200_search_bit_sequence(btle_b200_ctx *ctx, const int8_t *bit, size_t n, const int8_t *seq, size_t m);
/* crc24_core(bit_in, state_init_bit), btlelib.py:191-219: bit-serial CRC-24 LFSR, 24 result bits. */
int btle_b200_crc24_bits(btle_b200_ctx *ctx, const int8_t *bit_in, size_t n, const int8_t *state_init_bit,
                         int8_t *crc_bits_out);
/* scramble_core(bit_in, channel_number), btlelib.py:226-263: whitening of a bit array. */
int btle_b200_scramble_bits(btle_b200_ctx *ctx, const int8_t *bit_in, size_t n, int channel, int8_t *bit_out);

/* ---- the Python model's receiver, batched (BER sweep, BASELINE.json configs[3]) ----------------
 * btlelib.btle_rx(i, q, channel, crc_init_bits, aa_hex) (btlelib.py:414-541) for n_packets
 * windows of n_samples int16 samples each (n_samples a multiple of sps, n_samples/sps <= 2048):
 * symbol-spaced differential demod on each of the `sps` sample phases, exact 32-bit access
 * address search (first index), dewhitening from the PDU on, payload length from 6 (adv) or 5
 * bits, CRC-24 with the reference's clamp of the CRC position, first phase with CRC ok wins,
 * otherwise the values of the last phase that found the access address.  One warp per packet. */
typedef struct {
  int32_t start;         /* symbol index of the access address on the reported phase, -1 = never found */
  uint16_t n_pdu_bits;   /* len(pdu_bit)                                                              */
  uint8_t crc_ok;
  uint8_t phase;         /* sample_phase_idx as returned by btle_rx                                  */
  uint8_t payload_len;   /* num_byte_payload                                                         */
  uint8_t found;         /* 0: access address found on no phase; else 1 + the last phase it was found on
                            (== phase + 1 when crc_ok)                                                 */
  uint8_t pdu[70];       /* pdu_bit packed LSB first                                                 */
} btle_model_rx_rec;     /* 80 bytes */
int btle_b200_model_rx_batch_device(btle_b200_ctx *ctx, const int16_t *d_i, const int16_t *d_q, size_t n_packets,
                                    size_t n_samples, int sps, int channel, uint32_t crc_init, uint32_t access_addr,
                                    btle_model_rx_rec *d_out, void *cuda_stream);
int btle_b200_model_rx_batch(btle_b200_ctx *ctx, const int16_t *i, const int16_t *q, size_t n_packets, size_t n_samples,
                             int sps, int channel, uint32_t crc_init, uint32_t access_addr, btle_model_rx_rec *out);

/* ---- the Python model's receiver as a STREAMING mode over an 8-Msps capture (SURVEY.md §8f-3) -------------------
 * Input: interleaved int16 I,Q at 8 samples per symbol — the format `btle_ll -q` writes (firmware/btle_ll.c:50-51) and
 * python/test_btle_rx_by_captured_iq.py:71-78 reads.  btlelib.btle_rx works on one hand-cut window per packet; here the
 * windows are found on the GPU:
 *   1. sps8_hits_kernel: symbol-spaced differential bits on all 8 ABSOLUTE sample phases (phase = sample index mod 8)
 *      and every position where 32 of them equal the access address (HBM-bound, 4 bytes per sample);
 *   2. hits closer than BTLE_SPS8_MIN_PACKET_SYMBOLS symbols form one cluster (one packet seen on neighbouring
 *      phases); the first hit h of a cluster defines the window [w0, w0 + BTLE_SPS8_WINDOW), w0 = 8 (h / 8 -
 *      BTLE_SPS8_MARGIN_SYMBOLS) clamped to 0 — aligned to 8 samples, so the window's phases are the absolute ones;
 *      clusters whose window does not fit into the capture are dropped;
 *   3. the model receiver (8 phases, first CRC-ok phase wins; one warp per window) on every window, straight out of
 *      the capture;
 *   4. in time order, a window that starts inside the packet accepted before it is skipped.
 * rx == what btlelib.btle_rx returns for that window.  The CPU restatement oracle/btlelib_port.py follows the same four
 * steps and is pinned to the reference's btlelib window by window. */
#define BTLE_SPS8_WINDOW 3072              /* samples = 384 symbols: margin + AA + longest ADV PDU + CRC + slack        */
#define BTLE_SPS8_MARGIN_SYMBOLS 2
#define BTLE_SPS8_MIN_PACKET_SYMBOLS 72    /* access address + header + CRC                                           */
typedef struct {
  int64_t sample;          /* first sample of the access address on the reported phase (absolute, 8 Msps)            */
  int64_t window;          /* first sample of the window the model receiver ran on                                   */
  btle_model_rx_rec rx;
} btle_sps8_rec;           /* 96 bytes */
int btle_b200_rx_sps8(btle_b200_ctx *ctx, const int16_t *iq16, size_t n_samples, int channel, uint32_t crc_init,
                      uint32_t access_addr, btle_sps8_rec *out, size_t cap, size_t *n_out);
/* step 1 alone on a device-resident capture: *d_count (zeroed by the call) = number of hits, d_hits[0..min(count, cap)) =
 * their sample indices in no particular order; enqueued on cuda_stream, not synchronised */
int btle_b200_sps8_hits_device(btle_b200_ctx *ctx, const int16_t *d_iq16, size_t n_samples, uint32_t access_addr,
                               int64_t *d_hits, size_t cap, uint32_t *d_count, void *cuda_stream);

/* ---- BER flow of python/test_btle_ber.py, entirely on the device (BASELINE.json configs[3]) ----------------------
 * n_packets packets of the 39-byte ADV PDU of test_btle_ber.py:27 with random payload bits (:49): CRC-24, whitening,
 * the Python model's 8-sps modulator, add_freq_sampling_error(ppm) (btlelib.py:823-857), add_noise(snr) (:859-871),
 * np.int16() truncation [ber_synth_kernel] -> the model's receiver, one warp per packet [model_rx_batch_kernel] ->
 * the script's error accounting (:62-72: bit errors only in CRC-failed packets) [ber_score_kernel].  Randomness is a
 * hash of (seed, packet, sample), so a run is reproducible and packet k is the same whatever the batch size. */
typedef struct {
  uint64_t seed;
  float snr_db;
  float ppm;               /* 0, or -50..50 like test_btle_ber.py                                                  */
  int32_t channel;
  uint32_t crc_init;       /* as -k: 0x555555                                                                      */
  uint32_t access_addr;
  uint32_t reserved;
} btle_ber_cfg;
typedef struct {
  uint64_t packets, pkt_err, bit_err, bit_total, aa_miss;   /* aa_miss: CRC-failed packets whose access address was never found */
  double seconds;          /* device time of the run (CUDA events)                                                 */
} btle_ber_result;
int btle_b200_ber_run(btle_b200_ctx *ctx, const btle_ber_cfg *cfg, size_t n_packets, btle_ber_result *out);

/* ---- 16-bit IQ ingest (SURVEY.md §8f-3) ------------------------------------------------------------
 * bladeRF SC16Q11 samples are reduced to the receive chain's int8 exactly as the reference's
 * stream_callback does: out = (in >> shift) & 0xFF, shift = 4 (btle_rx.c:307-308).  Host buffers;
 * the conversion runs on the GPU, then the capture goes through the same path as btle_b200_rx(). */
int btle_b200_rx_iq16(btle_b200_ctx *ctx, const int16_t *iq16, size_t n_int16, int shift, const btle_stream_cfg *cfg,
                      btle_pkt_rec *out, size_t cap, size_t *n_out);

/* ---- wideband captures: exact integer channelizer (DESIGN.md §6.5) ------------------------------------------------
 * Input: ONE capture of n_samples complex samples, int8 interleaved I,Q (hackrf_transfer -r, UHD sc8) at
 * fs = 4 MHz * decim, centred on center_mhz.  Channel ch (f_ch = btle_b200_get_freq_by_channel_number(ch), offset
 * q = (f_ch - fc) / 1 MHz) is inside the band iff |q| + 1 <= fs/2 / 1 MHz.  For each output sample m < ceil(N / decim),
 * with x[n] = 0 outside [0, N) and c = (T-1)/2:
 *   acc[m] = sum_{t<T} x[m*decim + c - t] * H_q[t]                       complex, int32 (no overflow is possible)
 *   rot[m] = acc[m] * (-j)^((q*m) mod 4)                                  exact swap / negate of the int32 pair
 *   y[m]   = sat8((rot[m] + 2^(s-1)) >> s)  per component                 arithmetic shift, s = 0: no rounding term
 * H_q[t] = round(G * h[t] * exp(+j*2*pi*q*(t-c)/(4*decim))), h one odd-length, symmetric, real low-pass prototype per
 * decim (>= 50 dB from 1.25 MHz off the channel centre to fs/2, <= 1 dB droop within 0.6 MHz).  y is the channel at
 * 4 Msps with no delay: output sample m is wideband sample decim*m, so a record at (chunk, n0) lies at wideband sample
 * decim * (8192*chunk + n0).  Output layout [n_ch][out_stride_int8] int8 I,Q: the receiver's input format. */
typedef struct {
  int32_t decim;         /* 2..64: fs = 4 MHz * decim                                                           */
  int32_t center_mhz;    /* centre frequency of the capture, whole MHz                                          */
  int32_t out_shift;     /* -1 = default s (passband gain 1: output LSB = input LSB), else 0..31               */
  int32_t reserved;
} btle_wideband_cfg;
/* Host only (no context, no GPU): the T complex taps H_q[t] of `channel` as taps[2t] = Re, taps[2t+1] = Im, and the
 * shift `cfg` selects.  *n_taps = T always; BTLE_EOVERFLOW if cap (in complex taps) < T. */
int btle_b200_wideband_taps(const btle_wideband_cfg *cfg, int channel, int16_t *taps, size_t cap, size_t *n_taps,
                            int *out_shift);
/* Device buffers: d_wide (16-byte aligned, 2*n_samples int8) -> d_out (16-byte aligned) row i = channels[i] (host
 * array; duplicates allowed), out_stride_int8 a multiple of 16 and >= 2*ceil(n_samples/decim).  Enqueued on
 * cuda_stream, not synchronised. */
int btle_b200_channelize_device(btle_b200_ctx *ctx, const int8_t *d_wide, size_t n_samples, const btle_wideband_cfg *cfg,
                                const int32_t *channels, size_t n_ch, int8_t *d_out, size_t out_stride_int8, void *cuda_stream);
/* The same with host buffers (wide page-locked or pageable; out pageable is fine); returns when `out` is filled. */
int btle_b200_channelize(btle_b200_ctx *ctx, const int8_t *wide, size_t n_samples, const btle_wideband_cfg *cfg,
                         const int32_t *channels, size_t n_ch, int8_t *out, size_t out_stride_int8);
/* Channelize into context-owned scratch, then the receiver over all channels in one launch: channel i is
 * cfgs[i].channel, its records carry stream = i.  == btle_b200_rx_batch() over btle_b200_channelize()'s output
 * (n_int8 = 2*ceil(n_samples/decim) per channel), record for record; BTLE_EOVERFLOW as there. */
int btle_b200_rx_wideband(btle_b200_ctx *ctx, const int8_t *wide, size_t n_samples, const btle_wideband_cfg *cfg,
                          const btle_stream_cfg *cfgs, size_t n_ch, btle_pkt_rec *out, size_t cap, size_t *n_out);

/* ---- packet synthesiser (SURVEY.md §8f-1): the transmit PHY as a GPU kernel ---------------------
 * Integer GFSK modulation of n_packets packets given as air bytes (preamble, access address,
 * whitened PDU+CRC; bits LSB first), d_air [n_packets][max_bytes], d_nbytes [n_packets].
 *   sps == 4: gen_sample_from_phy_bit (host/btle-tools/src/btle_tx.c:1022-1063): +-1 impulses every
 *             4th sample, taps {2,11,32,53,60,53,32,11,2}, phase mod 1024, round(127 cos/sin).
 *             d_out_i receives interleaved int8 I,Q: [n_packets][2*(32*max_bytes+16)]; d_out_q unused.
 *   sps == 8: gfsk_modulation_fixed_point (python/btlelib.py:146-189): NRZ preceded by 17 samples of
 *             -1, 17 integer taps, >>1, phase mod 2048.  d_out_i / d_out_q: planar int8
 *             [n_packets][64*max_bytes+16].
 * Samples behind a packet's own 8*nbytes*sps+16 samples are written as 0.  Device pointers; enqueued
 * on cuda_stream, not synchronised. */
int btle_b200_tx_modulate_device(btle_b200_ctx *ctx, const uint8_t *d_air, const int32_t *d_nbytes, size_t n_packets,
                                 size_t max_bytes, int sps, int8_t *d_out_i, int8_t *d_out_q, void *cuda_stream);

/* ---- host-side functions the reference keeps next to receiver(): payload parsers, receiver_status and the
 *      connection follower (btle_b200/csrc/btle_host.cpp; no CUDA involved) ----------------------------------
 * Same argument meaning, return values (0 / -1, control opcode) and printed messages as
 *   int parse_adv_pdu_payload_byte(uint8_t*, int, ADV_PDU_TYPE, void*)   btle_rx.c:1564
 *   int parse_ll_pdu_payload_byte(uint8_t*, int, LL_PDU_TYPE, void*)     btle_rx.c:1741
 * `out` points at the struct matching the PDU type; layouts == the reference's typedefs (:1078-1210). */
typedef struct { uint8_t AdvA[6]; uint8_t Data[31]; } btle_adv_payload_0_2_4_6;      /* ADV_PDU_PAYLOAD_TYPE_0_2_4_6 */
typedef struct { uint8_t A0[6]; uint8_t A1[6]; } btle_adv_payload_1_3;               /* ADV_PDU_PAYLOAD_TYPE_1_3     */
typedef struct {
  uint8_t InitA[6]; uint8_t AdvA[6]; uint8_t AA[4]; uint32_t CRCInit; uint8_t WinSize;
  uint16_t WinOffset, Interval, Latency, Timeout; uint8_t ChM[5]; uint8_t Hop; uint8_t SCA;
} btle_adv_payload_5;                                                                /* ADV_PDU_PAYLOAD_TYPE_5       */
typedef struct { uint8_t payload_byte[40]; } btle_adv_payload_r;                     /* ADV_PDU_PAYLOAD_TYPE_R       */
typedef union { btle_adv_payload_0_2_4_6 t0246; btle_adv_payload_1_3 t13; btle_adv_payload_5 t5; btle_adv_payload_r r; } btle_adv_payload;
typedef struct { uint8_t Data[40]; } btle_ll_data_payload;                           /* LL_DATA_PDU_PAYLOAD_TYPE     */
typedef struct { uint8_t Opcode, WinSize; uint16_t WinOffset, Interval, Latency, Timeout, Instant; } btle_ll_ctrl_payload_0;
typedef struct { uint8_t Opcode; uint8_t ChM[5]; uint16_t Instant; } btle_ll_ctrl_payload_1;
typedef struct { uint8_t Opcode, ErrorCode; } btle_ll_ctrl_payload_2_7_13;
typedef struct { uint8_t Opcode; uint8_t Rand[8]; uint8_t EDIV[2]; uint8_t SKDm[8]; uint8_t IVm[4]; } btle_ll_ctrl_payload_3;
typedef struct { uint8_t Opcode; uint8_t SKDs[8]; uint8_t IVs[4]; } btle_ll_ctrl_payload_4;
typedef struct { uint8_t Opcode; } btle_ll_ctrl_payload_5_6_10_11;
typedef struct { uint8_t Opcode; uint8_t FeatureSet[8]; } btle_ll_ctrl_payload_8_9;
typedef struct { uint8_t Opcode, VersNr; uint16_t CompId, SubVersNr; } btle_ll_ctrl_payload_12;
typedef struct { uint8_t Opcode; uint8_t payload_byte[40]; } btle_ll_ctrl_payload_r;
typedef union {
  btle_ll_data_payload data; btle_ll_ctrl_payload_0 c0; btle_ll_ctrl_payload_1 c1; btle_ll_ctrl_payload_2_7_13 c2; btle_ll_ctrl_payload_3 c3;
  btle_ll_ctrl_payload_4 c4; btle_ll_ctrl_payload_5_6_10_11 c5; btle_ll_ctrl_payload_8_9 c8; btle_ll_ctrl_payload_12 c12; btle_ll_ctrl_payload_r r;
} btle_ll_payload;
int btle_b200_parse_adv_pdu_payload_byte(const uint8_t *payload_byte, int num_payload_byte, int pdu_type, void *adv_pdu_payload);
/* returns -1 (drop), else the control opcode (0 for data PDUs, where the reference's return value is undefined) */
int btle_b200_parse_ll_pdu_payload_byte(const uint8_t *payload_byte, int num_payload_byte, int pdu_type, void *ll_pdu_payload);
uint64_t btle_b200_get_freq_by_channel_number(int channel_number);                   /* btle_rx.c:1006 */
int btle_b200_chm_is_full_map(const uint8_t *chm);                                    /* btle_rx.c:2395 */

/* RECV_STATUS (btle_rx.c:1462-1471) — process-wide like the reference's global `receiver_status`: written by the
 * payload parsers (CONNECT_REQ, LL_CONNECTION_UPDATE_REQ, LL_CHANNEL_MAP_REQ) and by btle_b200_note_packet(),
 * read by btle_b200_receiver_controller(). */
typedef struct {
  int pkt_avaliable;
  int hop;               /* -1 until a CONNECT_REQ was parsed */
  int new_chm_flag;
  int interval;
  uint32_t access_addr;
  uint32_t crc_init;
  int crc_ok;            /* CRC verdict of the most recent counted packet (bool in the reference)            */
  uint8_t chm[5];
  uint8_t reserved;
} btle_receiver_status;
btle_receiver_status *btle_b200_receiver_status(void);
/* what receiver() does to receiver_status for every packet it counts (btle_rx.c:2320-2321) */
void btle_b200_note_packet(const btle_pkt_rec *rec);

/* receiver_controller (btle_rx.c:2403): the connection-following state machine, same signature.  Call it once per
 * processed chunk.  0 wait for a CRC-ok CONNECT_REQ with a full channel map -> 1 wait for the first CRC-ok data
 * packet -> 2 hop `interval - 7 ms` after the last mark -> 3 wait for a packet on the new channel, "skip" after
 * `interval - 4 ms`.  The reference reads the wall clock and retunes its radio from inside; here both are hooks,
 * so the same machine runs on sample time over per-channel captures (the btle_rx_b200 program does that). */
typedef struct {
  int64_t ts_us;
  char event[16];        /* track_start / track_drop / chan_change (btj_emit_hop, btle_json.c:132)               */
  int state_from, state_to, ch, freq_mhz;
  uint32_t access_addr, crc_init;
  int interval_us, hop;
  uint8_t chm[5];
} btle_hop_event;
typedef struct {
  int64_t (*now_us)(void *user);                          /* gettimeofday() of the reference                      */
  int (*set_freq)(void *user, uint64_t freq_hz);          /* board_set_freq(); non-zero = failure (-> returns -1) */
  void (*event)(void *user, const btle_hop_event *ev);    /* btj_emit_hop()                                       */
  void *user;
  int quiet_text;                                         /* quiet_text_flag: no "Hop: ..." lines on stdout       */
} btle_hop_hooks;
void btle_b200_set_hop_hooks(const btle_hop_hooks *hooks);
void btle_b200_hop_reset(void);                           /* state 0, receiver_status as main() initialises it    */
int btle_b200_receiver_controller(void *rf_dev, int verbose_flag, int *chan, uint32_t *access_addr, uint32_t *crc_init_internal);

/* ---- capture synthesiser (benchmark / test input; SURVEY.md §8d C2-C5) -----------------------------------
 * Fills n_streams device captures with a noise floor and one burst per `slot_samples` slot: an ADV_IND (TxAdd = 1,
 * AdvA = slot | stream << 32, 0..31 bytes of AdvData) on channels 37..39, an LL data PDU (0..27 bytes) elsewhere,
 * with the stream's access address / CRC init, CRC-24 + whitening + the btle_tx PHY (btle_tx.c:1022-1063) at
 * `amplitude`/127, added to the floor with saturation.  Every `corrupt_every`-th burst gets one flipped bit (its
 * CRC must fail), every `straddle_every`-th is placed ACROSS an 8192-sample chunk boundary (its decode needs the
 * look-ahead behind the chunk).  All randomness is a hash of (seed, stream, position): reproducible, no state.
 * d_truth (optional, [n_streams][n_slots]) receives what was sent. */
typedef struct {
  uint64_t seed;
  int32_t slot_samples;    /* >= 1600 (>= 3200 when straddle_every > 0)                                  */
  int32_t amplitude;       /* 0..127; 0 = no bursts                                                      */
  int32_t corrupt_every;   /* 0 = never                                                                  */
  int32_t straddle_every;  /* 0 = never, else >= 2                                                       */
  int32_t noise;           /* 0: floor of the reference capture (sigma 0.8 LSB, mean -0.3, clip -7..6);
                              1: full-scale uniform int8 (hot interferer); 2: none                       */
  int32_t reserved;
} btle_synth_cfg;
typedef struct {
  int64_t start_sample;    /* first sample of the preamble; the access address starts 39 samples later
                              at the receiver (32 preamble samples + modulator delay)                     */
  int32_t stream, slot;
  uint8_t n_air_bytes, corrupt, straddle, pdu_len;
  uint8_t pdu[44];         /* header + payload as sent (before CRC and whitening)                         */
} btle_synth_truth;        /* 64 bytes */
int btle_b200_synth_streams_device(btle_b200_ctx *ctx, int8_t *d_iq, size_t n_streams, size_t stream_stride_int8,
                                   size_t n_int8, const btle_stream_cfg *cfgs, const btle_synth_cfg *sc,
                                   btle_synth_truth *d_truth, size_t truth_cap, size_t *n_slots_out, void *cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* BTLE_B200_H */
