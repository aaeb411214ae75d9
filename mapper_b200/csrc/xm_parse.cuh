// xmapper_b200 — FASTA / FASTQ text to packed sequences on the device (xm_parse_reads).  Included by xm_capi.cu after xm_variants_fmt.cuh.
//
// One call parses the complete records at the start of a chunk of text:
//   xm_parse_nl_kernel<false>   per 4 KiB tile: the number of '\n' bytes (one ballot per warp per byte column of a 128-byte row);
//   cub exclusive scan           tile offsets;
//   xm_parse_nl_kernel<true>    the positions of the '\n' bytes, in order: line l of the text ends at line_end[l];
//   xm_parse_class_kernel        FASTA: header flags per line (then a cub scan gives every line its record, a cub select the header lines);
//   xm_parse_lines_kernel        bases per line of the parsed records, the line checks of FASTQ (marker, '+', quality length) and of FASTA
//                                (no text before the first header); cub scan: the base offset of every line;
//   xm_parse_rec_kernel          per record: its length and its number of --split-queries-past-size pieces; cub scan: the first piece;
//   xm_parse_piece_kernel        per piece: start, length, record, name length, words; cub scans: word offsets, name offsets;
//   xm_parse_pack_kernel         one warp per sequence, one thread per 16-bit word (four codes, no read-modify-write between threads), with
//                                the byte check of every base;
//   xm_parse_names_kernel        one warp per sequence: the header text, and "[start:end]" for a piece.
// Checks record the first bad byte (atomicMin over offset << 3 | kind) and the first bad line (atomicMin), so the host names both.
#pragma once

enum { PZ_OK = 0, PZ_BAD_BASE = 1, PZ_BAD_MARKER = 2, PZ_NO_PLUS = 3, PZ_QUAL_LEN = 4, PZ_BEFORE_HEADER = 5 };
static const int PZ_THREADS = 256;                 // 8 warps
static const int PZ_ROW = 128;                     // bytes one warp reads per step: 4 per lane
static const int PZ_ROWS = 4;                      // steps per warp
static const int PZ_TILE = PZ_THREADS / 32 * PZ_ROW * PZ_ROWS;   // 4096 bytes per block

struct PzErr { unsigned long long key, line; };    // key = byte offset << 3 | kind; ~0: no error

// ASCII -> 4-bit code of the 15 IUPAC letters of QV/Basepairs in either case; 0: not a base
__device__ __constant__ uint8_t XM_PZ_CODE[256] = {
  0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0,  0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0,
  0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0,  0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0,
  0, 1, 14, 2, 13, 0, 0, 4, 11, 0, 0, 12, 0, 3, 15, 0,   // @ A B C D E F G H I J K L M N O
  0, 0, 5, 6, 8, 0, 7, 9, 0, 10, 0, 0, 0, 0, 0, 0,       // P Q R S T U V W X Y Z
  0, 1, 14, 2, 13, 0, 0, 4, 11, 0, 0, 12, 0, 3, 15, 0,   // ` a .. o
  0, 0, 5, 6, 8, 0, 7, 9, 0, 10, 0, 0, 0, 0, 0, 0,       // p .. z
};

struct ParseD {
  const char* text; long long n;
  int fastq, split;
  const long long* line_end; int n_lines;            // line l = [line_end[l - 1] + 1, line_end[l]) (a '\r' before the end is dropped)
  const int* rec_line; int n_rec, lines_end;         // FASTA: header line of record r, rec_line[n_rec] = lines_end; FASTQ: 4r
  const int* line_rec;                               // FASTA: 1 + record of line l (0: before the first header)
  const long long* lbase;                            // bases of the parsed records before line l
  PzErr* err;
};

__device__ __forceinline__ long long pz_line_start(const ParseD& P, int l) { return l ? P.line_end[l - 1] + 1 : 0; }
__device__ __forceinline__ long long pz_line_stop(const ParseD& P, int l) {   // end without a trailing '\r'
  const long long s = pz_line_start(P, l), e = P.line_end[l];
  return (e > s && P.text[e - 1] == '\r') ? e - 1 : e;
}
__device__ __forceinline__ int pz_rec_line(const ParseD& P, int r) { return P.fastq ? 4 * r : P.rec_line[r]; }
__device__ __forceinline__ int pz_rec_line_end(const ParseD& P, int r) { return P.fastq ? 4 * r + 4 : P.rec_line[r + 1]; }
__device__ __forceinline__ void pz_fail(const ParseD& P, long long offset, int kind, int line) {
  atomicMin(&P.err->key, ((unsigned long long)offset << 3) | (unsigned long long)kind);
  atomicMin(&P.err->line, (unsigned long long)line);
}

// WRITE = false: tile_cnt[tile] = number of '\n' in the tile; WRITE = true: their positions from line_end[tile_off[tile]] on, in order
template <bool WRITE>
__global__ void __launch_bounds__(PZ_THREADS) xm_parse_nl_kernel(const char* text, long long n, unsigned int* tile_cnt, const unsigned int* tile_off, long long* line_end) {
  __shared__ unsigned int warp_cnt[PZ_THREADS / 32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long base = (long long)blockIdx.x * PZ_TILE + (long long)warp * PZ_ROW * PZ_ROWS;
  const unsigned lt = (1u << lane) - 1u;
  auto row_masks = [&](int row, unsigned m[4]) {
    const long long p = base + (long long)row * PZ_ROW + lane * 4;
    char c[4] = {0, 0, 0, 0};
    if (p + 3 < n) { const char4 v = *reinterpret_cast<const char4*>(text + p); c[0] = v.x; c[1] = v.y; c[2] = v.z; c[3] = v.w; }
    else for (int j = 0; j < 4; j++) if (p + j < n) c[j] = text[p + j];
    for (int j = 0; j < 4; j++) m[j] = __ballot_sync(0xffffffffu, c[j] == '\n');
  };
  unsigned int cnt = 0;
  for (int row = 0; row < PZ_ROWS; row++) { unsigned m[4]; row_masks(row, m); cnt += __popc(m[0]) + __popc(m[1]) + __popc(m[2]) + __popc(m[3]); }
  if (lane == 0) warp_cnt[warp] = cnt;
  __syncthreads();
  if (!WRITE) {
    if (threadIdx.x == 0) { unsigned int t = 0; for (int w = 0; w < PZ_THREADS / 32; w++) t += warp_cnt[w]; tile_cnt[blockIdx.x] = t; }
    return;
  }
  long long out = tile_off[blockIdx.x];
  for (int w = 0; w < warp; w++) out += warp_cnt[w];
  for (int row = 0; row < PZ_ROWS; row++) {
    unsigned m[4]; row_masks(row, m);
    // rank of byte (lane, j): the row's newlines in lanes below, then this lane's newlines in columns below j
    long long r = out + __popc(m[0] & lt) + __popc(m[1] & lt) + __popc(m[2] & lt) + __popc(m[3] & lt);
    const long long p = base + (long long)row * PZ_ROW + lane * 4;
    for (int j = 0; j < 4; j++) if ((m[j] >> lane) & 1u) line_end[r++] = p + j;
    out += __popc(m[0]) + __popc(m[1]) + __popc(m[2]) + __popc(m[3]);
  }
}

// FASTA: 1 where a line starts with '>'
__global__ void xm_parse_class_kernel(ParseD P, int* hdr_flag) {
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= P.n_lines) return;
  const long long s = pz_line_start(P, l);
  hdr_flag[l] = (s < P.line_end[l] && P.text[s] == '>') ? 1 : 0;
}

// bases per line of lines [0, lines_end) (0 for headers, '+' and quality lines) and the line checks; seq_bases has lines_end + 1 entries
__global__ void xm_parse_lines_kernel(ParseD P, long long* seq_bases) {
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l > P.lines_end) return;
  if (l == P.lines_end) { seq_bases[l] = 0; return; }
  const long long s = pz_line_start(P, l), e = pz_line_stop(P, l);
  long long nb = 0;
  if (P.fastq) {
    const int k = l & 3;
    if (k == 0 && (e == s || P.text[s] != '@')) pz_fail(P, s, PZ_BAD_MARKER, l);
    if (k == 1) nb = e - s;
    if (k == 2 && (e == s || P.text[s] != '+')) pz_fail(P, s, PZ_NO_PLUS, l);
    if (k == 3 && e - s != pz_line_stop(P, l - 2) - pz_line_start(P, l - 2)) pz_fail(P, s, PZ_QUAL_LEN, l);
  } else {
    const bool hdr = e > s && P.text[s] == '>';
    if (P.line_rec[l] == 0 && e > s) pz_fail(P, s, PZ_BEFORE_HEADER, l);
    else if (!hdr) nb = e - s;
  }
  seq_bases[l] = nb;
}

// per record: its number of pieces (M/SequenceSplitter.java:9-38: (len - 1) / split + 1 when split > 0)
__global__ void xm_parse_rec_kernel(ParseD P, long long* rec_pieces) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r > P.n_rec) return;
  if (r == P.n_rec) { rec_pieces[r] = 0; return; }
  const long long len = P.lbase[pz_rec_line_end(P, r)] - P.lbase[pz_rec_line(P, r)];
  rec_pieces[r] = (P.split > 0 && len > 0) ? (len - 1) / P.split + 1 : 1;
}

__device__ __forceinline__ int pz_digits(long long v) { int d = 1; while (v >= 10) { v /= 10; d++; } return d; }

struct PieceD { const long long* piece_off; long long* start; int32_t* len; int64_t* rec; long long* words; long long* name_len; };
// per record: its pieces [len * k / n, len * (k + 1) / n); a piece's name is the record's name + "[start:end]" when there are several
__global__ void xm_parse_piece_kernel(ParseD P, PieceD Q) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= P.n_rec) return;
  const long long len = P.lbase[pz_rec_line_end(P, r)] - P.lbase[pz_rec_line(P, r)];
  const long long s0 = Q.piece_off[r], np = Q.piece_off[r + 1] - s0;
  const int hl = pz_rec_line(P, r);
  const long long name_len = max(pz_line_stop(P, hl) - pz_line_start(P, hl) - 1, 0LL);
  for (long long k = 0; k < np; k++) {
    const long long a = len * k / np, b = len * (k + 1) / np, s = s0 + k;
    Q.start[s] = a; Q.len[s] = (int32_t)(b - a); Q.rec[s] = r; Q.words[s] = (b - a + 3) / 4;
    Q.name_len[s] = name_len + (np > 1 ? 3 + pz_digits(a) + pz_digits(b) : 0);
  }
}

struct PackD { const long long* start; const int32_t* len; const int64_t* rec; const int64_t* word_off; const int64_t* name_off; uint16_t* packed; char* names; long long n_seq; };

// the line of record-relative base `target` (absolute base index): the last line in [lo, hi) whose base offset is <= target
__device__ __forceinline__ int pz_find_line(const ParseD& P, int lo, int hi, long long target) {
  while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (P.lbase[mid] <= target) lo = mid; else hi = mid; }
  return lo;
}

__global__ void __launch_bounds__(256) xm_parse_pack_kernel(ParseD P, PackD K) {
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= K.n_seq) return;
  const long long s = warp;
  const int r = (int)K.rec[s], l0 = pz_rec_line(P, r), l1 = pz_rec_line_end(P, r);
  const long long b0 = P.lbase[l0] + K.start[s], len = K.len[s];
  uint16_t* out = K.packed + K.word_off[s];
  for (long long w = lane; 4 * w < len; w += 32) {
    long long t = b0 + 4 * w;
    int l = pz_find_line(P, l0, l1, t);
    unsigned word = 0;
    for (int j = 0; j < 4 && 4 * w + j < len; j++, t++) {
      while (t >= P.lbase[l + 1]) l++;
      const long long at = pz_line_start(P, l) + (t - P.lbase[l]);
      const uint8_t c = XM_PZ_CODE[(uint8_t)P.text[at]];
      if (!c) pz_fail(P, at, PZ_BAD_BASE, l);
      word |= (unsigned)c << (4 * j);
    }
    out[w] = (uint16_t)word;
  }
}

__global__ void __launch_bounds__(256) xm_parse_names_kernel(ParseD P, PackD K) {
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= K.n_seq) return;
  const long long s = warp;
  const int hl = pz_rec_line(P, (int)K.rec[s]);
  const long long a = pz_line_start(P, hl) + 1, nl = max(pz_line_stop(P, hl) - a, 0LL);
  char* out = K.names + K.name_off[s];
  for (long long i = lane; i < nl; i += 32) out[i] = P.text[a + i];
  if (lane == 0 && K.name_off[s + 1] - K.name_off[s] > nl) {   // a piece of a split record
    SamOut o; o.p = out + nl; o.n = 0;
    o.ch('['); o.num(K.start[s]); o.ch(':'); o.num(K.start[s] + K.len[s]); o.ch(']');
  }
}
