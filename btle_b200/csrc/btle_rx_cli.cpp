// btle_rx_b200 — btle_rx-compatible host program on top of the C-ABI (include/btle_b200.h).
//
// Keeps the option surface, text lines, NDJSON v1 events and pcap format of the reference's
// btle_rx (host/btle-tools/src/btle_rx.c: parse_commandline :1244-1458, receiver() sinks
// :2330-2389, pcap :110,:167-207; btle_json.c) so that its consumers (btle_cli: rx_proc.py:64-81,
// pcap_loader.py:93-144) keep working, but takes the IQ from a capture file instead of a radio and
// runs the whole receive chain on the GPU in one call.  Host-side work here is only what the
// reference does AFTER crc_check(): payload field re-ordering, the drop rules, the filters and the
// three sinks.
//
// Differences, on purpose:
//   * IQ source instead of an SDR (without one the program exits with status 1, the reference's "board failure"
//     code, :2586):
//       -i/--iq-file FILE        raw interleaved int8 (what rx_callback writes, btle_rx.c:531-540), '-' = stdin.  Read in
//                                64 MiB segments straight into page-locked memory and decoded while the next segment is
//                                being read (btle_b200_stream_*): the capture may be larger than host RAM or HBM.
//       -i FILE:CH[:AA[:CRCINIT]]  (repeatable) several captures, each with its own channel / access address / CRC
//                                init, decoded in ONE batched launch; packets are printed in time order.
//       --iq-dir DIR             DIR/ch00.bin .. DIR/ch39.bin, time-aligned captures of the BLE channels (missing
//                                files are skipped).  Without -o: like 40 -i entries.  With -o: see below.
//       --wideband FILE:RATE_MSPS:CENTER_MHZ   one int8 I,Q capture of the band at RATE_MSPS (a multiple of 4) centred on
//                                CENTER_MHZ (one SDR, hackrf_transfer -r / UHD sc8): every BLE channel inside the band is
//                                channelized on the GPU to 4 Msps (btle_b200_channelize), then handled exactly like
//                                --iq-dir, with and without -o; time stamps are on the 4 Msps channel time base.
//       --iq-txt FILE / --iq-sc16 FILE   text format of save_phy_sample (btle_rx.c:896-915) / int16 bladeRF samples.
//   * -o (hop) with --iq-dir: the reference retunes its ONE radio; here a virtual radio walks the per-channel captures
//     chunk by chunk with the reference's own state machine (btle_b200_receiver_controller == receiver_controller,
//     btle_rx.c:2403) on sample time: CONNECT_REQ on -c -> data channel (hop) -> hop every interval.  The decode for
//     every channel the radio could be on is done up front in two batched launches (advertising capture; then all 37
//     data captures with the connection's access address), the walk only picks what the radio would have seen.
//   * time stamps are sample time (4 Msps) from the start of the capture, not wall clock; in hop mode the state
//     machine's clock is the time at which a chunk (with its look-ahead) is complete.
#include <getopt.h>
#include <signal.h>
#include <unistd.h>

#include <algorithm>
#include <cerrno>

#include <climits>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "btle_b200.h"

namespace {

const char *ADV_NAME[16] = {"ADV_IND", "ADV_DIRECT_IND", "ADV_NONCONN_IND", "SCAN_REQ", "SCAN_RSP", "CONNECT_REQ",
                            "ADV_SCAN_IND", "RESERVED0", "RESERVED1", "RESERVED2", "RESERVED3", "RESERVED4",
                            "RESERVED5", "RESERVED6", "RESERVED7", "RESERVED8"};          // btle_rx.c:1153-1170
const char *LL_NAME[4] = {"LL_RESERVED", "LL_DATA1", "LL_DATA2", "LL_CTRL"};              // :1031-1036
const char *CTRL_NAME[15] = {"LL_CONNECTION_UPDATE_REQ", "LL_CHANNEL_MAP_REQ", "LL_TERMINATE_IND", "LL_ENC_REQ",
                             "LL_ENC_RSP", "LL_START_ENC_REQ", "LL_START_ENC_RSP", "LL_UNKNOWN_RSP", "LL_FEATURE_REQ",
                             "LL_FEATURE_RSP", "LL_PAUSE_ENC_REQ", "LL_PAUSE_ENC_RSP", "LL_VERSION_IND",
                             "LL_REJECT_IND", "LL_RESERVED"};                              // :1060-1076

struct Options {
  int chan = 37, gain = 6, lna = 32, amp = 0, verbose = 0, raw = 0, hop = 0, json = 0, quiet = 0, rssi = 0;
  uint32_t aa = 0x8E89BED6u, crc_init = 0x555555u, mask = 0xFFFFFFFFu;
  uint64_t freq_hz = 123;
  const char *pcap = nullptr, *iq_txt = nullptr, *iq_sc16 = nullptr, *iq_dir = nullptr, *iq_bin16 = nullptr, *wideband = nullptr;
  std::vector<std::string> iq_files;            // -i, possibly FILE:CH[:AA[:CRCINIT]]
  size_t segment_chunks = 4096;
  int filter_adva_set = 0;
  uint8_t filter_adva[6] = {0, 0, 0, 0, 0, 0};
  uint16_t filter_pdu_mask = 0xFFFF;
  int device = 0;
};

void usage() {
  printf(
      "Usage:\n"
      "    -h --help\n      Print this help screen\n"
      "    -i --iq-file FILE[:CH[:AA[:CRCINIT]]]\n      raw interleaved int8 I,Q capture at 4 Msps ('-' = stdin)   [this build: no SDR]\n"
      "      repeatable: several captures are decoded in one batch, each with its own channel / access address / CRC init\n"
      "       --iq-dir DIR\n      DIR/ch00.bin .. DIR/ch39.bin (time-aligned per-channel captures); with -o the connection is followed across them\n"
      "       --wideband FILE:RATE_MSPS:CENTER_MHZ\n      one int8 I,Q capture of the band (RATE_MSPS a multiple of 4, 8..256); every channel inside it is\n"
      "      channelized to 4 Msps on the GPU and decoded like --iq-dir (with -o the connection is followed across them)\n"
      "       --iq-bin16 FILE\n      interleaved int16 I,Q at 8 Msps (8 samples per symbol): a `btle_ll -q` capture; decoded with the 8-phase\n"
      "      CRC-select receiver of the reference's Python / Verilog model (first sample phase whose CRC is ok wins)\n"
      "       --segment-chunks N\n      chunks (16384 int8) per streamed segment of a single capture (default 4096 = 64 MiB)\n"
      "       --iq-txt FILE\n      capture in the text format written by save_phy_sample()\n"
      "       --iq-sc16 FILE\n      raw interleaved int16 I,Q (bladeRF SC16Q11); reduced with >>4 like btle_rx's bladeRF build\n"
      "    -c --chan\n      Channel number. default 37. valid range 0~39\n"
      "    -g --gain / -l --lnaGain / -b --amp / -f --freq_hz\n      accepted for compatibility; no radio is driven\n"
      "    -a --access\n      Access address. 4 bytes. Hex format (like 89ABCDEF). Default 8e89bed6\n"
      "    -k --crcinit\n      CRC init value. 3 bytes. Hex format (like 555555). Default 555555\n"
      "    -m --access_mask\n      Access address bit mask. Hex. Default ffffffff\n"
      "    -v --verbose / -r --raw / -o --hop\n"
      "    -s --filename\n      Store packets to pcap file (DLT 256, LE LL with PHDR)\n"
      "    -j --json / -Q --quiet-text / -R --rssi-est\n"
      "    -F --filter-adva AA:BB:CC:DD:EE:FF / -T --filter-pdu-type 0,3,4\n"
      "    -d --device N   CUDA device (default 0)\n");
}

int parse_mac(const char *s, uint8_t out[6]) {        // btle_rx.c:126-146
  if (!s) return -1;
  if (strchr(s, ':')) return sscanf(s, "%2hhx:%2hhx:%2hhx:%2hhx:%2hhx:%2hhx", &out[0], &out[1], &out[2], &out[3], &out[4], &out[5]) == 6 ? 0 : -1;
  if (strlen(s) != 12) return -1;
  for (int i = 0; i < 6; ++i)
    if (sscanf(s + 2 * i, "%2hhx", &out[i]) != 1) return -1;
  return 0;
}

int parse_pdu_csv(const char *s, uint16_t *mask) {    // btle_rx.c:149-165
  if (!s) return -1;
  uint16_t m = 0;
  const char *p = s;
  while (*p) {
    char *end;
    long v = strtol(p, &end, 10);
    if (end == p || v < 0 || v > 15) return -1;
    m |= (uint16_t)(1u << v);
    p = end;
    if (*p == ',') ++p; else if (*p) return -1;
  }
  if (!m) return -1;
  *mask = m;
  return 0;
}

[[noreturn]] void bad_args() {
  usage();
  exit(-1);                                           // btle_rx.c:1455-1457
}

Options parse_commandline(int argc, char **argv) {
  Options o;
  static struct option longopts[] = {
      {"help", no_argument, 0, 'h'}, {"chan", required_argument, 0, 'c'}, {"gain", required_argument, 0, 'g'},
      {"lnaGain", required_argument, 0, 'l'}, {"amp", no_argument, 0, 'b'}, {"access", required_argument, 0, 'a'},
      {"crcinit", required_argument, 0, 'k'}, {"verbose", no_argument, 0, 'v'}, {"raw", no_argument, 0, 'r'},
      {"freq_hz", required_argument, 0, 'f'}, {"access_mask", required_argument, 0, 'm'}, {"hop", no_argument, 0, 'o'},
      {"filename", required_argument, 0, 's'}, {"json", no_argument, 0, 'j'}, {"quiet-text", no_argument, 0, 'Q'},
      {"rssi-est", no_argument, 0, 'R'}, {"filter-adva", required_argument, 0, 'F'},
      {"filter-pdu-type", required_argument, 0, 'T'}, {"iq-file", required_argument, 0, 'i'},
      {"iq-txt", required_argument, 0, 1000}, {"iq-sc16", required_argument, 0, 1001}, {"device", required_argument, 0, 'd'},
      {"iq-dir", required_argument, 0, 1002}, {"segment-chunks", required_argument, 0, 1003}, {"iq-bin16", required_argument, 0, 1004},
      {"wideband", required_argument, 0, 1005}, {0, 0, 0, 0}};
  for (;;) {
    int idx = 0;
    const int c = getopt_long(argc, argv, "hc:g:l:ba:k:vrf:m:os:jQRF:T:i:d:", longopts, &idx);   // + i:, d:
    if (c == -1) break;
    char *endp;
    switch (c) {
      case 'v': o.verbose = 1; break;
      case 'r': o.raw = 1; break;
      case 'o': o.hop = 1; break;
      case 'c': o.chan = (int)strtol(optarg, &endp, 10); break;
      case 'g': o.gain = (int)strtol(optarg, &endp, 10); break;
      case 'l': o.lna = (int)strtol(optarg, &endp, 10); break;
      case 'b': o.amp = 1; break;
      case 'f': o.freq_hz = (uint64_t)strtol(optarg, &endp, 10); break;
      case 'a': o.aa = (uint32_t)strtol(optarg, &endp, 16); break;
      case 'm': o.mask = (uint32_t)strtol(optarg, &endp, 16); break;
      case 'k': o.crc_init = (uint32_t)strtol(optarg, &endp, 16); break;
      case 's': o.pcap = optarg; break;
      case 'j': o.json = 1; break;
      case 'Q': o.quiet = 1; break;
      case 'R': o.rssi = 1; break;
      case 'i': o.iq_files.push_back(optarg); break;
      case 1002: o.iq_dir = optarg; break;
      case 1004: o.iq_bin16 = optarg; break;
      case 1005: o.wideband = optarg; break;
      case 1003: o.segment_chunks = (size_t)strtoul(optarg, &endp, 10); break;
      case 1000: o.iq_txt = optarg; break;
      case 1001: o.iq_sc16 = optarg; break;
      case 'd': o.device = (int)strtol(optarg, &endp, 10); break;
      case 'F':
        if (parse_mac(optarg, o.filter_adva)) {
          printf("Invalid --filter-adva value: %s (expect AA:BB:CC:DD:EE:FF or 12 hex chars)\n", optarg);
          bad_args();
        }
        o.filter_adva_set = 1;
        break;
      case 'T':
        if (parse_pdu_csv(optarg, &o.filter_pdu_mask)) {
          printf("Invalid --filter-pdu-type value: %s (expect CSV of ints 0..15, e.g. 0,3,4)\n", optarg);
          bad_args();
        }
        break;
      default: bad_args();                            // 'h', '?', anything else
    }
  }
  if (o.chan < 0 || o.chan > 39) { printf("channel number must be within 0~%d!\n", 39); bad_args(); }   // :1432
  if (o.gain < 0 || o.gain > 62) { printf("rx gain must be within 0~%d!\n", 62); bad_args(); }            // :1437
  if (o.lna < 0 || o.lna > 40) { printf("lna gain must be within 0~%d!\n", 40); bad_args(); }            // :1442
  if (optind < argc) { printf("Error: unknown/extra arguments specified on command line!\n"); bad_args(); }
  return o;
}

uint64_t freq_by_channel(int ch) {                    // get_freq_by_channel_number, btle_rx.c:1006
  if (ch == 37) return 2402000000ull;
  if (ch == 38) return 2426000000ull;
  if (ch == 39) return 2480000000ull;
  if (ch <= 10) return 2404000000ull + (uint64_t)ch * 2000000ull;
  return 2428000000ull + (uint64_t)(ch - 11) * 2000000ull;
}

bool load_txt(const char *name, std::vector<int8_t> &iq) {   // numbers separated by ", " (save_phy_sample): one pass over the file
  FILE *f = fopen(name, "r");
  if (!f) { perror(name); return false; }
  std::vector<char> buf(1 << 20);
  long v = 0;
  bool in_num = false, neg = false;
  size_t n;
  while ((n = fread(buf.data(), 1, buf.size(), f)) > 0)
    for (size_t k = 0; k < n; ++k) {
      const char c = buf[k];
      if (c >= '0' && c <= '9') { v = v * 10 + (c - '0'); in_num = true; }
      else {
        if (in_num) { iq.push_back((int8_t)(neg ? -v : v)); v = 0; in_num = false; neg = false; }
        if (c == '-') neg = true;
      }
    }
  if (in_num) iq.push_back((int8_t)(neg ? -v : v));
  fclose(f);
  return true;
}

bool load_raw(const char *name, std::vector<int8_t> &iq) {
  FILE *f = strcmp(name, "-") ? fopen(name, "rb") : stdin;
  if (!f) { perror(name); return false; }
  if (f != stdin && fseek(f, 0, SEEK_END) == 0) {
    const long sz = ftell(f);
    fseek(f, 0, SEEK_SET);
    if (sz > 0) {
      iq.resize((size_t)sz);
      const size_t got = fread(iq.data(), 1, (size_t)sz, f);
      iq.resize(got);
      fclose(f);
      return true;
    }
  }
  char buf[1 << 16];
  size_t n;
  while ((n = fread(buf, 1, sizeof buf, f)) > 0) iq.insert(iq.end(), buf, buf + n);
  if (f != stdin) fclose(f);
  return true;
}

// ---- sinks ----------------------------------------------------------------------------------------
void put_be32(FILE *f, uint32_t v) { const uint8_t b[4] = {(uint8_t)(v >> 24), (uint8_t)(v >> 16), (uint8_t)(v >> 8), (uint8_t)v}; fwrite(b, 1, 4, f); }

FILE *pcap_open(const char *name) {                   // init_pcap_file + PCAP_HDR_TCPDUMP, btle_rx.c:110,:167
  FILE *f = fopen(name, "wb");
  if (!f) return nullptr;
  put_be32(f, 0xA1B2C3D4u);                           // magic, big-endian file
  const uint8_t ver[4] = {0, 2, 0, 4};
  fwrite(ver, 1, 4, f);
  put_be32(f, 0); put_be32(f, 0);                     // thiszone, sigfigs
  put_be32(f, 1500);                                  // snaplen 0x5DC
  put_be32(f, 256);                                   // DLT_BLUETOOTH_LE_LL_WITH_PHDR
  return f;
}

void pcap_write(FILE *f, double t, const uint8_t *pkt, int len, int ch, uint32_t aa, int rssi) {   // :184-207
  const uint32_t sec = (uint32_t)t, usec = (uint32_t)((t - sec) * 1e6);
  put_be32(f, sec); put_be32(f, usec);
  put_be32(f, 10 + 4 + (uint32_t)len); put_be32(f, 10 + 4 + (uint32_t)len);
  int8_t sig = -127;
  if (rssi != INT_MIN) sig = (int8_t)(rssi > 20 ? 20 : (rssi < -126 ? -126 : rssi));
  const uint8_t phdr[10] = {(uint8_t)ch, (uint8_t)sig, 0, 0, 0, 0, 0, 0, 1, 0};
  fwrite(phdr, 1, 10, f);
  const uint8_t aab[4] = {(uint8_t)aa, (uint8_t)(aa >> 8), (uint8_t)(aa >> 16), (uint8_t)(aa >> 24)};   // host order of the reference (LE)
  fwrite(aab, 1, 4, f);
  fwrite(pkt, 1, (size_t)len, f);
}

void hex(const uint8_t *b, int n) { for (int i = 0; i < n; ++i) printf("%02x", b[i]); }
void hex_rev(const uint8_t *b, int n) { for (int i = n - 1; i >= 0; --i) printf("%02x", b[i]); }   // fields printed MSB first
uint32_t le16(const uint8_t *p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8); }

// AdvA for the filter / JSON (extract_adv_a, :1720-1739): MSB-first; false = not available
bool adv_a(const uint8_t *p, int type, uint8_t out[6]) {
  int off;
  if (type == 0 || type == 2 || type == 4 || type == 6 || type == 1 || type == 3) off = 0;
  else if (type == 5) off = 6;
  else return false;
  for (int i = 0; i < 6; ++i) out[i] = p[off + 5 - i];
  return true;
}
void print_adv_payload(const uint8_t *p, int type, int plen, int crc_bad) {     // print_adv_pdu_payload, :2131-2185
  if (type == 0 || type == 2 || type == 4 || type == 6) {
    printf("AdvA:"); hex_rev(p, 6);
    printf(" Data:"); hex(p + 6, plen - 6);
  } else if (type == 1 || type == 3) {
    printf("A0:"); hex_rev(p, 6);
    printf(" A1:"); hex_rev(p + 6, 6);
  } else if (type == 5) {
    printf("InitA:"); hex_rev(p, 6);
    printf(" AdvA:"); hex_rev(p + 6, 6);
    printf(" AA:"); hex_rev(p + 12, 4);
    const uint32_t crcinit = ((uint32_t)p[16] << 16) | ((uint32_t)p[17] << 8) | p[18];
    printf(" CRCInit:%06x WSize:%02x WOffset:%04x Itrvl:%04x Ltncy:%04x Timot:%04x", crcinit, p[19], le16(p + 20), le16(p + 22), le16(p + 24), le16(p + 26));
    printf(" ChM:"); hex_rev(p + 28, 5);
    printf(" Hop:%d SCA:%d", p[33] & 0x1F, (p[33] >> 5) & 7);
  } else {
    printf("Byte:"); hex(p, plen);
  }
  printf(" CRC%d\n", crc_bad);
}

void print_ll_payload(const uint8_t *p, int llid, int op, int plen, int crc_bad) {   // print_ll_pdu_payload, :2018-2129
  if (plen == 0) { printf("CRC%d\n", crc_bad); return; }
  if (llid != 3) {
    printf("LL_Data:"); hex(p, plen);
  } else if (op == 0) {
    printf("Op%02x(%s) WSize:%02x WOffset:%04x Itrvl:%04x Ltncy:%04x Timot:%04x Inst:%04x", op, CTRL_NAME[op], p[1], le16(p + 2), le16(p + 4), le16(p + 6), le16(p + 8), le16(p + 10));
  } else if (op == 1) {
    printf("Op%02x(%s)", op, CTRL_NAME[op]); printf(" ChM:"); hex_rev(p + 1, 5); printf(" Inst:%04x", le16(p + 6));
  } else if (op == 2 || op == 7 || op == 13) {
    printf("Op%02x(%s) Err:%02x", op, CTRL_NAME[op], p[1]);
  } else if (op == 3) {
    printf("Op%02x(%s)", op, CTRL_NAME[op]);
    printf(" Rand:"); hex_rev(p + 1, 8); printf(" EDIV:"); hex_rev(p + 9, 2);
    printf(" SKDm:"); hex_rev(p + 11, 8); printf(" IVm:"); hex_rev(p + 19, 4);
  } else if (op == 4) {
    printf("Op%02x(%s)", op, CTRL_NAME[op]); printf(" SKDs:"); hex_rev(p + 1, 8); printf(" IVs:"); hex_rev(p + 9, 4);
  } else if (op == 5 || op == 6 || op == 10 || op == 11) {
    printf("Op%02x(%s)", op, CTRL_NAME[op]);
  } else if (op == 8 || op == 9) {
    printf("Op%02x(%s)", op, CTRL_NAME[op]); printf(" FteurSet:"); hex_rev(p + 1, 8);
  } else if (op == 12) {
    printf("Op%02x(%s) Ver:%02x CompId:%04x SubVer:%04x", op, CTRL_NAME[op], p[1], le16(p + 2), le16(p + 4));
  } else {
    printf("Op%02x(%s)", op, CTRL_NAME[op > 13 ? 14 : op]); printf(" Byte:"); hex(p + 1, plen - 1);
  }
  printf(" CRC%d\n", crc_bad);
}

void json_hex(const uint8_t *b, int n) { putchar('"'); hex(b, n); putchar('"'); }
void json_status(double ts, const char *event, const Options &o) {               // btj_emit_status
  printf("{\"v\":1,\"t\":\"status\",\"ts\":%.6f,\"event\":\"%s\",\"board\":\"B200-file\",\"ch\":%d,\"freq_hz\":%llu,\"gain\":%d,\"lna\":%d,\"amp\":%d,\"filter_adva\":",
         ts, event, o.chan, (unsigned long long)o.freq_hz, o.gain, o.lna, o.amp);
  if (o.filter_adva_set) printf("\"%02x:%02x:%02x:%02x:%02x:%02x\"", o.filter_adva[0], o.filter_adva[1], o.filter_adva[2], o.filter_adva[3], o.filter_adva[4], o.filter_adva[5]);
  else printf("null");
  printf(",\"msg\":null}\n");
  fflush(stdout);
}

int rssi_from_mag(unsigned mag_sum) {                 // btle_rx.c:2244-2249
  double mean = (double)mag_sum / 128.0;
  if (mean < 1.0) mean = 1.0;
  int r = (int)(20.0 * log10(mean / 256.0) - 50.0);
  if (r < -127) r = -127;
  if (r > 20) r = 20;
  return r;
}

// ---- what receiver() does with a counted packet after crc_check(): filters, sinks (btle_rx.c:2318-2389) -----------
struct Sinks {
  const Options &o;
  FILE *pcap = nullptr;
  int pkt_count = 0;
  double t_prev = 0.0;
  explicit Sinks(const Options &opt) : o(opt) {}

  void packet(const btle_pkt_rec &r, double t) {
    const uint8_t *b = r.bytes;
    const int ch = r.channel;
    const uint32_t aa = r.access_addr;
    const bool adv = (ch == 37 || ch == 38 || ch == 39);                        // :2202
    if (r.flags & BTLE_REC_REJECTED) {                                          // :2291-2298, only with -v
      int type, tx, rx, plen;
      btle_b200_parse_adv_pdu_header_byte(b, &type, &tx, &rx, &plen);
      printf("XXXus PktBAD Ch%d AA:%08x ", ch, aa);
      printf("ADV_PDU_t%d:%s T%d R%d PloadL%d ", type, ADV_NAME[type], tx, rx, plen);
      printf("Error: ADV payload length should be 6~37!\n");
      return;
    }
    ++pkt_count;                                                                // :2274 / :2319
    btle_b200_note_packet(&r);                                                  // receiver_status.crc_ok, :2320-2321
    const int time_diff = (int)llround((t - t_prev) * 1e6);
    t_prev = t;
    const int rssi = o.rssi ? rssi_from_mag(r.mag_sum) : INT_MIN;
    if (r.flags & 1) {                                                          // raw, :2271-2286
      const long sec = (long)t;
      printf("%ld.%06ld Pkt%d Ch%d AA:%08x Raw:", sec, (long)((t - sec) * 1e6), pkt_count, ch, aa);
      hex(b, 42);
      printf("\n");
      return;
    }
    const int crc_bad = r.crc_bad;
    if (adv) {
      int type, tx, rx, plen;
      btle_b200_parse_adv_pdu_header_byte(b, &type, &tx, &rx, &plen);
      if (!(o.filter_pdu_mask & (1u << (type & 15)))) return;                   // :2332-2334
      btle_adv_payload parsed;
      if (btle_b200_parse_adv_pdu_payload_byte(b + 2, plen, type, &parsed)) return;   // :2336-2339 (also feeds receiver_status)
      uint8_t a[6];
      const bool has_a = adv_a(b + 2, type, a);
      if (o.filter_adva_set && has_a && memcmp(a, o.filter_adva, 6)) return;    // :2345-2348
      if (pcap) pcap_write(pcap, t, b, plen + 2, ch, aa, rssi);                 // :2361-2362
      if (!o.quiet) {
        printf("%07dus Pkt%03d Ch%d AA:%08x ", time_diff, pkt_count, ch, aa);
        printf("ADV_PDU_t%d:%s T%d R%d PloadL%d ", type, ADV_NAME[type], tx, rx, plen);
        print_adv_payload(b + 2, type, plen, crc_bad);
      }
      if (o.json) {                                                             // btj_emit_pkt_adv
        printf("{\"v\":1,\"t\":\"pkt\",\"ts\":%.6f,\"pkt\":%d,\"ch\":%d,\"aa\":\"%08x\",\"crc_ok\":%s,\"kind\":\"adv\",\"pdu_type\":%d,\"pdu_name\":\"%s\"",
               t, pkt_count, ch, aa, crc_bad ? "false" : "true", type, ADV_NAME[type]);
        printf(",\"tx_add\":%d,\"rx_add\":%d,\"plen\":%d,\"adv_a\":", tx, rx, plen);
        if (has_a) printf("\"%02x:%02x:%02x:%02x:%02x:%02x\"", a[0], a[1], a[2], a[3], a[4], a[5]); else printf("null");
        printf(",\"payload_hex\":"); json_hex(b + 2, plen);
        if (rssi == INT_MIN) printf(",\"rssi_est\":null"); else printf(",\"rssi_est\":%d", rssi);
        printf("}\n");
      }
    } else {
      int llid, nesn, sn, md, plen;
      btle_b200_parse_ll_pdu_header_byte(b, &llid, &nesn, &sn, &md, &plen);
      btle_ll_payload parsed;
      const int op = btle_b200_parse_ll_pdu_payload_byte(b + 2, plen, llid, &parsed);
      if (op < 0) return;                                                       // :2350-2353
      if (o.filter_adva_set) return;                                            // :2355-2357
      if (pcap) pcap_write(pcap, t, b, plen + 2, ch, aa, rssi);
      if (!o.quiet) {
        printf("%07dus Pkt%03d Ch%d AA:%08x ", time_diff, pkt_count, ch, aa);
        printf("LL_PDU_t%d:%s NESN%d SN%d MD%d PloadL%d ", llid, LL_NAME[llid], nesn, sn, md, plen);
        print_ll_payload(b + 2, llid, op, plen, crc_bad);
      }
      if (o.json) {                                                             // btj_emit_pkt_data
        printf("{\"v\":1,\"t\":\"pkt\",\"ts\":%.6f,\"pkt\":%d,\"ch\":%d,\"aa\":\"%08x\",\"crc_ok\":%s,\"kind\":\"data\",\"ll_pdu_type\":%d,\"ll_pdu_name\":\"%s\"",
               t, pkt_count, ch, aa, crc_bad ? "false" : "true", llid, LL_NAME[llid]);
        printf(",\"nesn\":%d,\"sn\":%d,\"md\":%d,\"plen\":%d,\"payload_hex\":", nesn, sn, md, plen);
        json_hex(b + 2, plen);
        if (rssi == INT_MIN) printf(",\"rssi_est\":null"); else printf(",\"rssi_est\":%d", rssi);
        printf("}\n");
      }
    }
  }
};

double rec_time(const btle_pkt_rec &r) { return ((double)r.chunk * 8192.0 + r.n0) / 4.0e6; }   // sample time of the access address

volatile sig_atomic_t g_stop = 0;
void on_sigint(int) { g_stop = 1; }                                             // btle_rx.c:100-104

struct Capture { std::string file; int chan; uint32_t aa, crc_init; std::vector<int8_t> *mem = nullptr; };

// a per-channel capture: the file, or (--wideband) the channel already channelized into memory
bool load_capture(const Capture &c, std::vector<int8_t> &iq) {
  if (c.mem) { iq.swap(*c.mem); return true; }
  return load_raw(c.file.c_str(), iq);
}

// --wideband FILE:RATE_MSPS:CENTER_MHZ -> chan_iq[ch] = 4 Msps capture of every channel inside the band, one Capture each
// (advertising access address / CRC init on 37..39, -a / -k elsewhere, as for --iq-dir)
int load_wideband(btle_b200_ctx *ctx, const Options &o, std::vector<std::vector<int8_t>> &chan_iq, std::vector<Capture> &caps) {
  const std::string spec = o.wideband;
  const size_t c2 = spec.rfind(':'), c1 = c2 == std::string::npos || c2 == 0 ? std::string::npos : spec.rfind(':', c2 - 1);
  char *e1 = nullptr, *e2 = nullptr;
  const long rate = c1 == std::string::npos ? 0 : strtol(spec.c_str() + c1 + 1, &e1, 10);
  const long center = c1 == std::string::npos ? 0 : strtol(spec.c_str() + c2 + 1, &e2, 10);
  if (c1 == std::string::npos || *e1 != ':' || *e2 || rate < 8 || rate > 256 || rate % 4) {
    printf("--wideband expects FILE:RATE_MSPS:CENTER_MHZ with RATE_MSPS a multiple of 4 in 8..256: %s\n", o.wideband);
    return BTLE_EINVAL;
  }
  std::vector<int8_t> wide;
  if (!load_raw(spec.substr(0, c1).c_str(), wide)) return BTLE_EINVAL;
  const btle_wideband_cfg cfg{(int32_t)(rate / 4), (int32_t)center, -1, 0};
  std::vector<int32_t> chans;
  for (int ch = 0; ch < 40; ++ch)
    if (std::labs((long)(freq_by_channel(ch) / 1000000) - center) + 1 <= 2 * cfg.decim) chans.push_back(ch);
  if (chans.empty()) { printf("no BLE channel inside %ld Msps around %ld MHz\n", rate, center); return BTLE_EINVAL; }
  const size_t n = wide.size() / 2, width = 2 * ((n + cfg.decim - 1) / cfg.decim), stride = (width + 15) & ~size_t(15);
  std::vector<int8_t> out(stride * chans.size());
  const int rc = btle_b200_channelize(ctx, wide.data(), n, &cfg, chans.data(), chans.size(), out.data(), stride);
  if (rc) { printf("btle_b200_channelize: %s (%s)\n", btle_b200_strerror(rc), btle_b200_last_error(ctx)); return rc; }
  for (size_t i = 0; i < chans.size(); ++i) {
    const int ch = chans[i];
    chan_iq[ch].assign(out.begin() + i * stride, out.begin() + i * stride + width);
    const bool adv = ch >= 37;
    caps.push_back(Capture{o.wideband, ch, adv ? 0x8E89BED6u : o.aa, adv ? 0x555555u : o.crc_init, &chan_iq[ch]});
  }
  return BTLE_OK;
}

// "FILE[:CH[:AA[:CRCINIT]]]"
Capture parse_capture(const std::string &spec, const Options &o) {
  Capture c{spec, o.chan, o.aa, o.crc_init};
  std::vector<std::string> parts;
  size_t pos = 0;
  for (;;) {
    const size_t q = spec.find(':', pos);
    parts.push_back(spec.substr(pos, q == std::string::npos ? q : q - pos));
    if (q == std::string::npos) break;
    pos = q + 1;
  }
  // a ':' inside a path: only trailing fields that look like numbers are taken as parameters
  size_t nfield = 0;
  while (nfield < 3 && parts.size() > 1 + nfield) {
    const std::string &f = parts[parts.size() - 1 - nfield];
    if (f.empty() || f.find_first_not_of("0123456789abcdefABCDEF") != std::string::npos) break;
    ++nfield;
  }
  // fields are CH, then AA, then CRCINIT: with 1 field it is CH, with 2 CH:AA, with 3 CH:AA:CRCINIT
  const size_t first = parts.size() - nfield;
  if (nfield >= 1) c.chan = (int)strtol(parts[first].c_str(), nullptr, 10);
  if (nfield >= 2) c.aa = (uint32_t)strtoul(parts[first + 1].c_str(), nullptr, 16);
  if (nfield >= 3) c.crc_init = (uint32_t)strtoul(parts[first + 2].c_str(), nullptr, 16);
  c.file.clear();
  for (size_t k = 0; k < first; ++k) c.file += (k ? ":" : "") + parts[k];
  return c;
}

int cfg_flags(const Options &o) { return (o.rssi ? BTLE_CFG_RSSI : 0) | (o.verbose ? BTLE_CFG_REPORT_REJECTED : 0); }

// rx_batch with a capacity that is grown once if the library asks
int rx_batch_grow(btle_b200_ctx *ctx, const int8_t *iq, size_t ns, size_t stride, size_t n, const btle_stream_cfg *cfgs,
                  std::vector<btle_pkt_rec> &recs) {
  size_t cap = ns * (n / BTLE_CHUNK_INT8) * 4 + 1024, got = 0;
  int rc = 0;
  for (int attempt = 0; attempt < 2; ++attempt) {
    recs.resize(cap);
    rc = btle_b200_rx_batch(ctx, iq, ns, stride, n, cfgs, recs.data(), cap, &got);
    if (rc != BTLE_EOVERFLOW) break;
    cap = got;
  }
  recs.resize(rc ? 0 : got);
  return rc;
}

// ---- hop mode: a virtual radio over per-channel captures (receiver_controller semantics) -------------------------
struct HopRun {
  const Options *o;
  int64_t now = 0;
  int retunes = 0;
};
int64_t hop_now(void *u) { return static_cast<HopRun *>(u)->now; }
int hop_set_freq(void *u, uint64_t) { ++static_cast<HopRun *>(u)->retunes; return 0; }
void hop_event(void *u, const btle_hop_event *e) {                              // btj_emit_hop, btle_json.c:132-160
  const HopRun *h = static_cast<HopRun *>(u);
  if (!h->o->json) return;
  printf("{\"v\":1,\"t\":\"hop\",\"ts\":%.6f,\"event\":\"%s\",\"state_from\":%d,\"state_to\":%d,\"ch\":%d,\"freq_mhz\":%d,"
         "\"aa\":\"%08x\",\"crc_init\":\"%06x\",\"interval_us\":%d,\"hop\":%d,\"chm\":\"%02x%02x%02x%02x%02x\"}\n",
         (double)e->ts_us / 1e6, e->event, e->state_from, e->state_to, e->ch, e->freq_mhz, e->access_addr, e->crc_init & 0xFFFFFFu,
         e->interval_us, e->hop, e->chm[0], e->chm[1], e->chm[2], e->chm[3], e->chm[4]);
}
// time at which chunk k and its look-ahead are complete: what the reference's wall clock shows when it runs receiver() on it
int64_t chunk_done_us(long long k) { return (int64_t)(((k + 1) * 8192ll + BTLE_LOOKAHEAD_INT8 / 2) / 4); }

}  // namespace

int main(int argc, char **argv) {
  printf("BLE sniffer (B200 offline receive chain; option surface of btle_rx by Xianjun Jiao)\n\n");
  Options o = parse_commandline(argc, argv);
  if (o.freq_hz == 123) o.freq_hz = freq_by_channel(o.chan);                    // btle_rx.c:2558
  if (!o.quiet)
    printf("Cmd line input: chan %d, freq %ldMHz, access addr %08x, crc init %06x raw %d verbose %d rx %ddB (%s) file=%s\n", o.chan,
           (long)(o.freq_hz / 1000000), o.aa, o.crc_init, o.raw, o.verbose, o.gain, "B200-file", o.pcap ? o.pcap : "(null)");
  Sinks sinks(o);
  if (o.pcap) {
    if (!o.quiet) printf("will store packets to: %s\n", o.pcap);
    sinks.pcap = pcap_open(o.pcap);
    if (!sinks.pcap) { perror(o.pcap); return 1; }
  }
  if (o.json) json_status(0.0, "start", o);
  if (o.iq_files.empty() && !o.iq_txt && !o.iq_sc16 && !o.iq_dir && !o.iq_bin16 && !o.wideband) {
    printf("open_board: no SDR support in this build; give a capture with -i/--iq-file\n");
    if (o.json) json_status(0.0, "stop", o);
    return 1;                                                                   // btle_rx.c:2586
  }
  struct sigaction sa;
  memset(&sa, 0, sizeof sa);
  sa.sa_handler = on_sigint;
  sigaction(SIGINT, &sa, nullptr);
  sigaction(SIGTERM, &sa, nullptr);

  btle_b200_bind_host_numa(o.device, nullptr);                                  // page-locked buffers next to the GPU
  btle_b200_ctx *ctx = nullptr;
  int rc = btle_b200_create(&ctx, o.device);
  if (rc) { printf("btle_b200_create: %s\n", btle_b200_strerror(rc)); return 1; }
  btle_b200_hop_reset();
  auto fail = [&](const char *what) {
    printf("%s: %s (%s)\n", what, btle_b200_strerror(rc), btle_b200_last_error(ctx));
    btle_b200_destroy(ctx);
    return 1;
  };
  double t_end = 0.0;

  // ---------------------------------------------------------------------------------------------------------------
  std::vector<Capture> caps;
  for (const std::string &f : o.iq_files) caps.push_back(parse_capture(f, o));
  if (o.iq_dir) {
    for (int ch = 0; ch < 40; ++ch) {
      char name[512];
      snprintf(name, sizeof name, "%s/ch%02d.bin", o.iq_dir, ch);
      if (access(name, R_OK) != 0) continue;
      const bool adv = ch >= 37;
      caps.push_back(Capture{name, ch, adv ? 0x8E89BED6u : o.aa, adv ? 0x555555u : o.crc_init});
    }
    if (caps.empty()) { printf("no chNN.bin capture found in %s\n", o.iq_dir); btle_b200_destroy(ctx); return 1; }
  }
  // per-channel captures of the band: --iq-dir files or the channels of --wideband; the paths below do not tell them apart
  std::vector<std::vector<int8_t>> wide_ch(40);
  if (o.wideband && !o.iq_dir && load_wideband(ctx, o, wide_ch, caps) != BTLE_OK) { btle_b200_destroy(ctx); return 1; }
  const char *per_channel = o.iq_dir ? o.iq_dir : o.wideband;
  for (const Capture &c : caps)
    if (c.chan < 0 || c.chan > 39) { printf("channel number must be within 0~%d!\n", 39); btle_b200_destroy(ctx); return 1; }

  if (o.iq_bin16) {
    // ---- 8 samples per symbol: the Python / Verilog model's receiver, streaming over the capture -------------------------
    std::vector<int8_t> raw;
    if (!load_raw(o.iq_bin16, raw)) { btle_b200_destroy(ctx); return 1; }
    const size_t n_samples = raw.size() / 4;
    std::vector<btle_sps8_rec> recs(n_samples / 576 + 16);
    size_t n = 0;
    rc = btle_b200_rx_sps8(ctx, reinterpret_cast<const int16_t *>(raw.data()), n_samples, o.chan, o.crc_init, o.aa, recs.data(), recs.size(), &n);
    if (rc) return fail("btle_b200_rx_sps8");
    const bool adv = (o.chan == 37 || o.chan == 38 || o.chan == 39);
    for (size_t i = 0; i < n && !g_stop; ++i) {
      const btle_model_rx_rec &m = recs[i].rx;
      if (!m.found || m.n_pdu_bits < 16) continue;         // no header decoded: nothing the sinks could show
      btle_pkt_rec r;
      memset(&r, 0, sizeof r);
      const int have = m.n_pdu_bits / 8;                    // header + payload bytes that were decoded (CRC clamp, btlelib.py:488-490)
      memcpy(r.bytes, m.pdu, (size_t)std::min(have, 39));
      const int plen = std::min(have - 2, (int)(r.bytes[1] & (adv ? 0x3F : 0x1F)));
      r.bytes[1] = (uint8_t)((r.bytes[1] & (adv ? 0xC0 : 0xE0)) | plen);
      r.channel = (uint8_t)o.chan; r.access_addr = o.aa; r.flags = adv ? 2 : 0;
      r.crc_bad = m.crc_ok ? 0 : 1;
      r.n_bytes = (uint8_t)(plen + 5);
      sinks.packet(r, (double)recs[i].sample / 8.0e6);
    }
    t_end = (double)n_samples / 8.0e6;
  } else if (o.hop && per_channel) {
    // ---- connection following over per-channel captures ---------------------------------------------------------
    std::vector<std::vector<int8_t>> iq(40);
    size_t n = SIZE_MAX;
    for (const Capture &c : caps) {
      if (!load_capture(c, iq[c.chan])) { btle_b200_destroy(ctx); return 1; }
      n = std::min(n, iq[c.chan].size());
    }
    if (iq[o.chan].empty()) { printf("no capture of the start channel %d in %s\n", o.chan, per_channel); btle_b200_destroy(ctx); return 1; }
    const long long nchunks = (long long)(n / BTLE_CHUNK_INT8);
    HopRun run{&o};
    btle_hop_hooks hooks{hop_now, hop_set_freq, hop_event, &run, o.quiet};
    btle_b200_set_hop_hooks(&hooks);
    int chan = o.chan;
    uint32_t aa = o.aa, crc_internal = btle_b200_crc_init_reorder(o.crc_init);
    // pass A: the start channel with the command line's access address, all chunks
    std::vector<btle_pkt_rec> recs;
    btle_stream_cfg cfg0{o.chan, o.aa, o.mask, o.crc_init, o.raw, cfg_flags(o)};
    rc = rx_batch_grow(ctx, iq[o.chan].data(), 1, n, n, &cfg0, recs);
    if (rc) return fail("btle_b200_rx_batch");
    size_t ri = 0;
    long long k = 0;
    for (; k < nchunks && !g_stop; ++k) {
      for (; ri < recs.size() && recs[ri].chunk == k; ++ri) sinks.packet(recs[ri], rec_time(recs[ri]));
      run.now = chunk_done_us(k);
      if (btle_b200_receiver_controller(nullptr, o.verbose, &chan, &aa, &crc_internal) != 0) break;   // :2655-2658
      if (chan != o.chan) { ++k; break; }                    // track start: the radio now sits on a data channel
    }
    if (chan != o.chan && k < nchunks) {
      // pass B: every data channel from chunk k on, with the connection's parameters, one batched launch
      const btle_receiver_status *st = btle_b200_receiver_status();
      const size_t off = (size_t)k * BTLE_CHUNK_INT8, n2 = n - off, stride = (n2 + 15) & ~size_t(15);
      std::vector<int> chan_of;
      for (int c = 0; c < 37; ++c) if (!iq[c].empty()) chan_of.push_back(c);
      std::vector<int8_t> stage(stride * chan_of.size());
      std::vector<btle_stream_cfg> cfgs;
      for (size_t s_ = 0; s_ < chan_of.size(); ++s_) {
        memcpy(stage.data() + s_ * stride, iq[chan_of[s_]].data() + off, n2);
        cfgs.push_back(btle_stream_cfg{chan_of[s_], st->access_addr, o.mask, st->crc_init, o.raw, cfg_flags(o)});
      }
      std::vector<btle_pkt_rec> data;
      rc = rx_batch_grow(ctx, stage.data(), chan_of.size(), stride, n2, cfgs.data(), data);
      if (rc) return fail("btle_b200_rx_batch");
      // index: first record of every (stream, chunk)
      std::vector<size_t> first(chan_of.size() * (size_t)(nchunks - k) + 1, 0);
      {
        size_t p = 0;
        for (size_t b = 0; b + 1 < first.size(); ++b) {
          const int s_ = (int)(b / (size_t)(nchunks - k)), c = (int)(b % (size_t)(nchunks - k));
          while (p < data.size() && (data[p].stream < s_ || (data[p].stream == s_ && data[p].chunk < c))) ++p;
          first[b] = p;
        }
        first.back() = data.size();
      }
      std::vector<int> stream_of(40, -1);
      for (size_t s_ = 0; s_ < chan_of.size(); ++s_) stream_of[chan_of[s_]] = (int)s_;
      for (; k < nchunks && !g_stop; ++k) {
        const int s_ = stream_of[chan];
        if (s_ >= 0) {
          const size_t b = (size_t)s_ * (size_t)(nchunks - (long long)(off / BTLE_CHUNK_INT8)) + (size_t)(k - (long long)(off / BTLE_CHUNK_INT8));
          for (size_t p = first[b]; p < first[b + 1]; ++p) {
            btle_pkt_rec r = data[p];
            r.chunk += (int32_t)(off / BTLE_CHUNK_INT8);
            sinks.packet(r, rec_time(r));
          }
        }
        run.now = chunk_done_us(k);
        if (btle_b200_receiver_controller(nullptr, o.verbose, &chan, &aa, &crc_internal) != 0) break;
      }
    }
    btle_b200_set_hop_hooks(nullptr);
    t_end = (double)(n / 2) / 4.0e6;
  } else if (caps.size() > 1 || (caps.size() == 1 && per_channel)) {
    // ---- several captures: one batched launch, packets in time order ------------------------------------------------
    std::vector<std::vector<int8_t>> iq(caps.size());
    size_t n = SIZE_MAX;
    for (size_t s_ = 0; s_ < caps.size(); ++s_) {
      if (!load_capture(caps[s_], iq[s_])) { btle_b200_destroy(ctx); return 1; }
      n = std::min(n, iq[s_].size());
    }
    const size_t stride = (n + 15) & ~size_t(15);
    std::vector<int8_t> stage(stride * caps.size());
    std::vector<btle_stream_cfg> cfgs;
    for (size_t s_ = 0; s_ < caps.size(); ++s_) {
      memcpy(stage.data() + s_ * stride, iq[s_].data(), n);
      iq[s_] = std::vector<int8_t>();
      cfgs.push_back(btle_stream_cfg{caps[s_].chan, caps[s_].aa, o.mask, caps[s_].crc_init, o.raw, cfg_flags(o)});
    }
    std::vector<btle_pkt_rec> recs;
    rc = rx_batch_grow(ctx, stage.data(), caps.size(), stride, n, cfgs.data(), recs);
    if (rc) return fail("btle_b200_rx_batch");
    std::stable_sort(recs.begin(), recs.end(), [](const btle_pkt_rec &a, const btle_pkt_rec &b) {
      const long long ta = (long long)a.chunk * 8192 + a.n0, tb = (long long)b.chunk * 8192 + b.n0;
      return ta < tb;                                          // ties keep (stream, chunk, n0) order
    });
    for (const btle_pkt_rec &r : recs) { if (g_stop) break; sinks.packet(r, rec_time(r)); }
    t_end = (double)(n / 2) / 4.0e6;
  } else if (o.iq_txt || o.iq_sc16) {
    // ---- whole-file formats ----------------------------------------------------------------------------------------
    std::vector<int8_t> iq;
    if (o.iq_sc16 ? !load_raw(o.iq_sc16, iq) : !load_txt(o.iq_txt, iq)) { btle_b200_destroy(ctx); return 1; }
    btle_stream_cfg cfg{o.chan, o.aa, o.mask, o.crc_init, o.raw, cfg_flags(o)};
    const size_t n_iq = o.iq_sc16 ? iq.size() / 2 : iq.size();          // int8 values after the optional reduction
    size_t cap = (n_iq / BTLE_CHUNK_INT8) * 4 + 1024, n = 0;
    std::vector<btle_pkt_rec> recs;
    for (int attempt = 0; attempt < 2; ++attempt) {
      recs.resize(cap);
      if (o.iq_sc16) rc = btle_b200_rx_iq16(ctx, reinterpret_cast<const int16_t *>(iq.data()), n_iq, 4, &cfg, recs.data(), cap, &n);   // btle_rx.c:307-308
      else rc = btle_b200_rx(ctx, iq.data(), iq.size(), &cfg, recs.data(), cap, &n);
      if (rc != BTLE_EOVERFLOW) break;
      cap = n;
    }
    if (rc) return fail("btle_b200_rx");
    for (size_t i = 0; i < n && !g_stop; ++i) sinks.packet(recs[i], rec_time(recs[i]));
    t_end = (double)(n_iq / 2) / 4.0e6;
  } else {
    // ---- one raw capture, streamed: read() straight into page-locked segments while the GPU decodes the previous one ----
    const Capture c = caps[0];
    FILE *f = strcmp(c.file.c_str(), "-") ? fopen(c.file.c_str(), "rb") : stdin;
    if (!f) { perror(c.file.c_str()); btle_b200_destroy(ctx); return 1; }
    btle_stream_cfg cfg{c.chan, c.aa, o.mask, c.crc_init, o.raw, cfg_flags(o)};
    btle_b200_stream *st = nullptr;
    rc = btle_b200_stream_open(ctx, &cfg, o.segment_chunks, &st);
    if (rc) return fail("btle_b200_stream_open");
    std::vector<btle_pkt_rec> recs(65536);
    size_t total = 0;
    const int fd = fileno(f);
    bool eof = false;
    while (!eof && !g_stop) {
      int8_t *buf; size_t space;
      btle_b200_stream_acquire(st, &buf, &space);
      const ssize_t got = read(fd, buf, std::min(space, size_t(8) << 20));
      if (got < 0) { if (errno == EINTR) continue; perror("read"); break; }
      if (got == 0) { eof = true; break; }
      total += (size_t)got;
      size_t n = 0;
      rc = btle_b200_stream_commit(st, (size_t)got, recs.data(), recs.size(), &n);
      if (rc) { btle_b200_stream_close(st); return fail("btle_b200_stream_commit"); }
      for (size_t i = 0; i < n; ++i) sinks.packet(recs[i], rec_time(recs[i]));
      if (n) fflush(stdout);
    }
    for (;;) {
      size_t n = 0;
      rc = btle_b200_stream_finish(st, recs.data(), recs.size(), &n);
      for (size_t i = 0; i < n; ++i) sinks.packet(recs[i], rec_time(recs[i]));
      if (rc != BTLE_EOVERFLOW) break;
    }
    btle_b200_stream_close(st);
    if (rc) return fail("btle_b200_stream_finish");
    if (f != stdin) fclose(f);
    t_end = (double)(total / 2) / 4.0e6;
  }

  fflush(stdout);
  if (!o.quiet) printf("Exit main loop ...\n");                                 // :2664
  if (o.json) json_status(t_end, "stop", o);
  if (sinks.pcap) fclose(sinks.pcap);
  btle_b200_destroy(ctx);
  return 0;
}
