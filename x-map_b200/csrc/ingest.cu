// Text ingest of the rating files (SURVEY.md 8(f) #4: clean / split on the device + the 4-column text reader).
// Replaces the line reading of LocalContext.textFile (text mode: lines end at \n, \r\n or a lone \r; whitespace-only
// lines are skipped) and the per-line work of BaselinerClean.parse_data (baselinerClean.py:38-56): str.split() into
// uid iid rating timestamp, iid + label, float() of the rating and of the timestamp.
//   ingest_mask_kernel / ingest_offset_kernel : the byte pass.  16-byte loads, one 16-bit terminator mask per chunk,
//                                              then the masks (1/8 of the bytes) are expanded into int64 line ends.
//   ingest_parse_kernel                       : one warp per 32 lines; the warp's byte span is staged in shared
//                                              memory, each lane tokenises and parses one line.
//   ingest_rank_*                             : boundary flags over LSD-sorted id words -> dense ranks.
//   ingest_first_kernel                       : first in-period line of every user and of every (user, item) pair
//                                              (the dict insertion order of filter_data).
//   ingest_item_*                             : the per-item string tests of encode.item_codes.
//   ingest_train_keys_kernel                  : the record order of BaselinerSplit.split_data.
#include "common.cuh"

namespace xmap {

constexpr int ING_BLOCK = 256;
constexpr int ING_WARPS = ING_BLOCK / 32;
constexpr int ING_SPAN = 2048;                 // staged bytes per warp (32 lines of up to 64 B); longer spans read HBM
constexpr int ING_WORDS = XMAP_INGEST_ID_MAX / 8;

// Python's str.split() whitespace restricted to ASCII (\r only survives before \n here, where it is dropped anyway)
__device__ __forceinline__ bool is_ws(uint8_t c) { return c == ' ' || (c >= 9 && c <= 13) || (c >= 0x1c && c <= 0x1f); }

// one bit per byte of a 32-bit word that equals c (SIMD byte compare, then the byte flags gathered into 4 bits)
__device__ __forceinline__ uint32_t byte_bits(uint32_t w, uint32_t c4) {
    const uint32_t y = __vcmpeq4(w, c4) & 0x01010101u;
    return (y | y >> 7 | y >> 14 | y >> 21) & 0xfu;
}

// bit b: byte pos+b ends a line.  `next` = the byte after the chunk (0 past the end; the buffer is zero padded)
__device__ __forceinline__ uint32_t chunk_mask(uint4 v, uint8_t next, long long pos, long long size) {
    const uint32_t mn = byte_bits(v.x, 0x0a0a0a0au) | byte_bits(v.y, 0x0a0a0a0au) << 4 |
                        byte_bits(v.z, 0x0a0a0a0au) << 8 | byte_bits(v.w, 0x0a0a0a0au) << 12;
    const uint32_t mr = byte_bits(v.x, 0x0d0d0d0du) | byte_bits(v.y, 0x0d0d0d0du) << 4 |
                        byte_bits(v.z, 0x0d0d0d0du) << 8 | byte_bits(v.w, 0x0d0d0d0du) << 12;
    const uint32_t before_n = mn >> 1 | (next == '\n' ? 1u << 15 : 0u);
    uint32_t m = mn | (mr & ~before_n);
    if (pos + 16 > size) m &= (1u << (uint32_t)max(size - pos, 0ll)) - 1u;
    return m;
}

__global__ void __launch_bounds__(ING_BLOCK) ingest_mask_kernel(const uint4 *__restrict__ buf, long long size,
                                                                uint16_t *__restrict__ masks, int32_t *__restrict__ block_cnt) {
    const long long nch = (size + 15) / 16;
    const long long c = (long long)blockIdx.x * ING_BLOCK + threadIdx.x;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (c < nch) v = buf[c];
    // the byte after this chunk: the first byte of the next lane's chunk, or one load at a warp's edge
    uint8_t next = (uint8_t)__shfl_down_sync(0xffffffffu, v.x & 0xff, 1);
    if (lane_id() == 31 && 16 * c + 16 < size) next = reinterpret_cast<const uint8_t *>(buf)[16 * c + 16];
    const uint32_t m = c < nch ? chunk_mask(v, next, 16 * c, size) : 0;
    if (c < nch) masks[c] = (uint16_t)m;
    int cnt = __popc(m);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, off);
    __shared__ int ws[ING_WARPS];
    if (lane_id() == 0) ws[threadIdx.x >> 5] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        int s = 0;
        for (int k = 0; k < ING_WARPS; ++k) s += ws[k];
        block_cnt[blockIdx.x] = s;
    }
}

__global__ void __launch_bounds__(ING_BLOCK) ingest_offset_kernel(const uint16_t *__restrict__ masks, long long nch,
                                                                  const int64_t *__restrict__ block_off,
                                                                  int64_t *__restrict__ offs) {
    const long long c = (long long)blockIdx.x * ING_BLOCK + threadIdx.x;
    uint32_t m = c < nch ? masks[c] : 0;
    const int cnt = __popc(m);
    int incl = cnt;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, incl, off);
        if (lane_id() >= off) incl += y;
    }
    __shared__ int ws[ING_WARPS];
    if (lane_id() == 31) ws[threadIdx.x >> 5] = incl;
    __syncthreads();
    int base = 0;
    for (int k = 0; k < (int)(threadIdx.x >> 5); ++k) base += ws[k];
    long long o = block_off[blockIdx.x] + base + incl - cnt;
    while (m) {
        const int b = __ffs(m) - 1;
        m &= m - 1;
        offs[o++] = 16 * c + b;
    }
}

__constant__ double c_pow10[23] = {1e0, 1e1, 1e2, 1e3, 1e4, 1e5, 1e6, 1e7, 1e8, 1e9, 1e10, 1e11,
                                   1e12, 1e13, 1e14, 1e15, 1e16, 1e17, 1e18, 1e19, 1e20, 1e21, 1e22};

// [+-]?(d+(.d*)?|.d+)([eE][+-]?d+)? with at most 15 significant digits and a decimal exponent within +-22: the value
// is m * 10^e or m / 10^-e with m < 2^53 and 10^|e| exact, ONE correctly rounded operation, so it equals Python's
// correctly rounded float().  Anything else is refused (false).
__device__ bool parse_number(const uint8_t *p, int a, int b, double *out) {
    int k = a;
    bool neg = false;
    if (k < b && (p[k] == '+' || p[k] == '-')) { neg = p[k] == '-'; ++k; }
    unsigned long long m = 0;
    int nd = 0, pend = 0, dexp = 0, ndig = 0;
    bool frac = false;
    for (; k < b; ++k) {
        const uint8_t c = p[k];
        if (c == '.' && !frac) { frac = true; continue; }
        if (c < '0' || c > '9') break;
        ++ndig;
        if (frac) --dexp;
        const int d = c - '0';
        if (d == 0) {
            if (m) ++pend;                     // a zero after the first significant digit: held back
        } else {
            nd += pend + 1;
            if (nd > 15) return false;
            for (; pend > 0; --pend) m *= 10;
            m = m * 10 + d;
        }
    }
    if (ndig == 0) return false;
    if (k < b && (p[k] == 'e' || p[k] == 'E')) {
        ++k;
        int es = 1;
        if (k < b && (p[k] == '+' || p[k] == '-')) { es = p[k] == '-' ? -1 : 1; ++k; }
        int ed = 0, ev = 0;
        for (; k < b && p[k] >= '0' && p[k] <= '9'; ++k) {
            ++ed;
            if (ev < 100000) ev = ev * 10 + (p[k] - '0');
        }
        if (ed == 0) return false;
        dexp += es * ev;
    }
    if (k != b) return false;
    if (m == 0) { *out = neg ? -0.0 : 0.0; return true; }
    const int e = dexp + pend;
    if (e < -22 || e > 22) return false;
    double v = (double)m;
    v = e >= 0 ? __dmul_rn(v, c_pow10[e]) : __ddiv_rn(v, c_pow10[-e]);
    *out = neg ? -v : v;
    return true;
}

__device__ __forceinline__ uint8_t label_byte(unsigned long long l0, unsigned long long l1, int k) {
    return (uint8_t)((k < 8 ? l0 >> (56 - 8 * k) : l1 >> (56 - 8 * (k - 8))) & 0xff);
}

__global__ void __launch_bounds__(ING_BLOCK) ingest_parse_kernel(
    const uint8_t *__restrict__ buf, const int64_t *__restrict__ offs, long long n, unsigned long long lab0,
    unsigned long long lab1, int lab_len, double ts_min, double ts_max, long long ld, uint8_t *__restrict__ status,
    double *__restrict__ rating, double *__restrict__ ts, unsigned long long *__restrict__ uw,
    uint8_t *__restrict__ ulen, unsigned long long *__restrict__ iw, uint8_t *__restrict__ ilen) {
    __shared__ uint8_t span[ING_WARPS][ING_SPAN];
    const int wid = threadIdx.x >> 5, lane = lane_id();
    const long long first = ((long long)blockIdx.x * ING_WARPS + wid) * 32;
    if (first >= n) return;
    const long long last = min(first + 31, n - 1);
    const long long s_lo = first == 0 ? 0 : offs[first - 1] + 1, s_hi = offs[last];
    const long long j = first + lane;
    const uint8_t *base = buf;
    long long sub = 0;
    if (s_hi - s_lo <= ING_SPAN) {
        for (long long k = s_lo + lane; k < s_hi; k += 32) span[wid][k - s_lo] = buf[k];
        base = span[wid];
        sub = s_lo;
    }
    __syncwarp();
    if (j >= n) return;
    const long long lo = (j == 0 ? 0 : offs[j - 1] + 1) - sub;
    const int len = (int)min((long long)(offs[j] - sub - lo), (long long)0x7fffffff);
    const uint8_t *p = base + lo;

    int tb[4], te[4], ntok = 0;
    bool in = false;
    int st = XMAP_INGEST_OK;
    for (int k = 0; k < len; ++k) {
        const uint8_t c = p[k];
        if (c == 0) { st = XMAP_INGEST_NUL; break; }
        if (c >= 0x80) { st = XMAP_INGEST_NON_ASCII; break; }
        if (is_ws(c)) {
            if (in) { if (ntok < 4) te[ntok] = k; ++ntok; in = false; }
        } else if (!in) {
            in = true;
            if (ntok < 4) tb[ntok] = k;
        }
    }
    if (st == XMAP_INGEST_OK && in) { if (ntok < 4) te[ntok] = len; ++ntok; }
    double r = __longlong_as_double(0x7ff8000000000000ll), t = r;    // NaN: never in a period
    if (st == XMAP_INGEST_OK) {
        if (ntok == 0) st = XMAP_INGEST_BLANK;
        else if (ntok < 4) st = XMAP_INGEST_FEW_FIELDS;
        else if (!parse_number(p, tb[3], te[3], &t)) st = XMAP_INGEST_BAD_TIME;
        else if (!(t >= ts_min && t <= ts_max)) st = XMAP_INGEST_TIME_RANGE;
        else if (!parse_number(p, tb[2], te[2], &r)) st = XMAP_INGEST_BAD_RATING;
        else if (te[0] - tb[0] > XMAP_INGEST_ID_MAX) st = XMAP_INGEST_UID_LONG;
        else if (te[1] - tb[1] + lab_len > XMAP_INGEST_ID_MAX) st = XMAP_INGEST_IID_LONG;
    }
    status[j] = (uint8_t)st;
    if (st != XMAP_INGEST_OK) {
        rating[j] = __longlong_as_double(0x7ff8000000000000ll);
        ts[j] = rating[j];
        ulen[j] = 0;
        ilen[j] = 0;
        return;                                // the id words stay zero (the caller zeroes them)
    }
    rating[j] = r;
    ts[j] = t;
    const int ul = te[0] - tb[0], rl = te[1] - tb[1], il = rl + lab_len;
    ulen[j] = (uint8_t)ul;
    ilen[j] = (uint8_t)il;
    // ids as big-endian 64-bit words, zero padded: byte order = string order, top bit 0 (ASCII)
    for (int w = 0; w * 8 < ul; ++w) {
        unsigned long long v = 0;
#pragma unroll
        for (int b = 0; b < 8; ++b) {
            const int k = 8 * w + b;
            v = (v << 8) | (k < ul ? p[tb[0] + k] : 0u);
        }
        uw[w * ld + j] = v;
    }
    for (int w = 0; w * 8 < il; ++w) {
        unsigned long long v = 0;
#pragma unroll
        for (int b = 0; b < 8; ++b) {
            const int k = 8 * w + b;
            const uint8_t c = k < rl ? p[tb[1] + k] : (k < il ? label_byte(lab0, lab1, k - rl) : 0);
            v = (v << 8) | c;
        }
        iw[w * ld + j] = v;
    }
}

// flag[p] = 1 where the id at sorted position p differs from the one before it
__global__ void __launch_bounds__(ING_BLOCK) ingest_rank_flags_kernel(const unsigned long long *__restrict__ words,
                                                                      long long ld, int nw, const int64_t *__restrict__ perm,
                                                                      long long n, int32_t *__restrict__ flag) {
    const long long p = (long long)blockIdx.x * ING_BLOCK + threadIdx.x;
    if (p >= n) return;
    int f = p == 0;
    if (!f) {
        const long long a = perm[p], b = perm[p - 1];
        for (int w = 0; w < nw && !f; ++w) f = words[w * ld + a] != words[w * ld + b];
    }
    flag[p] = f;
}

// rank[perm[p]] = csum[p] - 1 (csum = inclusive scan of flag); rep[rank] = the first line of the rank in sorted order
__global__ void __launch_bounds__(ING_BLOCK) ingest_rank_scatter_kernel(const int64_t *__restrict__ perm,
                                                                        const int32_t *__restrict__ flag,
                                                                        const int64_t *__restrict__ csum, long long n,
                                                                        int32_t *__restrict__ rank, int64_t *__restrict__ rep) {
    const long long p = (long long)blockIdx.x * ING_BLOCK + threadIdx.x;
    if (p >= n) return;
    const int32_t r = (int32_t)(csum[p] - 1);
    rank[perm[p]] = r;
    if (flag[p]) rep[r] = perm[p];
}

// Over the records in clean order (in-period first, then by user, item; stable): the first in-period line of every
// user (atomicMin) and, for every kept record, the first in-period line of its (user, item) pair = the start of its run.
__global__ void __launch_bounds__(ING_BLOCK) ingest_first_kernel(const int32_t *__restrict__ user,
                                                                 const int32_t *__restrict__ item,
                                                                 const double *__restrict__ ts,
                                                                 const int64_t *__restrict__ order,
                                                                 const uint8_t *__restrict__ keep, long long n,
                                                                 double t_lo, double t_hi, int32_t *__restrict__ first_user,
                                                                 int32_t *__restrict__ pair_first) {
    const long long p = (long long)blockIdx.x * ING_BLOCK + threadIdx.x;
    if (p >= n) return;
    const long long r = order[p];
    const double t = ts[r];
    if (!(t >= t_lo && t < t_hi)) return;
    const int u = user[r], i = item[r];
    atomicMin(first_user + u, (int)r);
    if (!keep[r]) return;
    long long q = p;
    while (q > 0) {
        const long long r2 = order[q - 1];
        const double t2 = ts[r2];
        if (user[r2] != u || item[r2] != i || !(t2 >= t_lo && t2 < t_hi)) break;
        --q;
    }
    pair_first[r] = (int32_t)order[q];
}

__device__ __forceinline__ int id_byte(const unsigned long long *w, long long ld, long long line, int k) {
    return (int)((w[(k >> 3) * ld + line] >> (56 - 8 * (k & 7))) & 0xff);
}

// s[-2:] of every item as a 16-bit key ordered like the strings (a 1-character id keeps its byte in the high half)
__device__ __forceinline__ int suffix_key(const unsigned long long *w, long long ld, long long line, int L) {
    return L >= 2 ? (id_byte(w, ld, line, L - 2) << 8) | id_byte(w, ld, line, L - 1) : id_byte(w, ld, line, 0) << 8;
}

__global__ void __launch_bounds__(ING_BLOCK) ingest_item_suffix_kernel(const unsigned long long *__restrict__ iw,
                                                                       long long ld, const uint8_t *__restrict__ ilen,
                                                                       const int64_t *__restrict__ rep, int32_t n_items,
                                                                       uint8_t *__restrict__ present) {
    const int i = blockIdx.x * ING_BLOCK + threadIdx.x;
    if (i >= n_items) return;
    const long long line = rep[i];
    present[suffix_key(iw, ld, line, ilen[line])] = 1;
}

// Items in ascending id order.  prefix_new[i] = iid[:2] differs from item i-1's (the caller scans it into the prefix
// rank), dom_code = rank of iid[-2:] among `labels` (sorted suffix keys), contains bit d = label d in iid, has_S / has_T.
__global__ void __launch_bounds__(ING_BLOCK) ingest_item_codes_kernel(
    const unsigned long long *__restrict__ iw, long long ld, const uint8_t *__restrict__ ilen,
    const int64_t *__restrict__ rep, int32_t n_items, const int32_t *__restrict__ labels, int32_t n_labels,
    int32_t *__restrict__ prefix_new, uint8_t *__restrict__ dom_code, uint8_t *__restrict__ contains,
    bool *__restrict__ has_S, bool *__restrict__ has_T) {
    const int i = blockIdx.x * ING_BLOCK + threadIdx.x;
    if (i >= n_items) return;
    const long long line = rep[i];
    const int L = ilen[line];
    prefix_new[i] = i == 0 || (iw[line] >> 48) != (iw[rep[i - 1]] >> 48);
    const int sk = suffix_key(iw, ld, line, L);
    int dc = 0;
    for (int d = 0; d < n_labels; ++d) if (labels[d] == sk) dc = d;
    bool s = false, t = false;
    uint32_t ct = 0;
    int prev = 0;
    for (int k = 0; k < L; ++k) {
        const int c = id_byte(iw, ld, line, k);
        s |= prev == 'S' && c == ':';
        t |= prev == 'T' && c == ':';
        for (int d = 0; d < n_labels; ++d) {
            const int a = labels[d] >> 8, b = labels[d] & 0xff;
            if (b ? (prev == a && c == b) : c == a) ct |= 1u << d;
        }
        prev = c;
    }
    dom_code[i] = (uint8_t)dc;
    contains[i] = (uint8_t)ct;
    has_S[i] = s;
    has_T[i] = t;
}

// Train order of BaselinerSplit.split_data: key = group << 58 | user position << 26 | sub, -1 for a test record.
//   group (per user): 0 non-overlap source, 1 non-overlap target, 2 both, 3 rest, 4 test user
//   sub: 0, or for a test user's target-list record 1 + its draw rank in random.sample (test record if not drawn)
__global__ void __launch_bounds__(ING_BLOCK) ingest_train_keys_kernel(const int32_t *__restrict__ user,
                                                                      const int32_t *__restrict__ item,
                                                                      const int8_t *__restrict__ grp,
                                                                      const int32_t *__restrict__ upos,
                                                                      const bool *__restrict__ has_S,
                                                                      const int32_t *__restrict__ srank, long long n,
                                                                      int64_t *__restrict__ key) {
    const long long r = (long long)blockIdx.x * ING_BLOCK + threadIdx.x;
    if (r >= n) return;
    const int u = user[r];
    const long long g = grp[u];
    long long sub = 0;
    if (g == 4 && !has_S[item[r]]) {
        if (srank[r] < 0) { key[r] = -1; return; }
        sub = 1 + srank[r];
    }
    key[r] = g << 58 | (long long)upos[u] << 26 | sub;
}

inline unsigned blocks_of(long long n) { return (unsigned)((n + ING_BLOCK - 1) / ING_BLOCK); }

}  // namespace xmap

using namespace xmap;

extern "C" int xmap_ingest_line_masks(const void *buf, int64_t size, uint16_t *masks, int32_t *block_cnt, void *stream) {
    if (size < 0) return fail_msg("xmap_ingest_line_masks: negative size");
    if ((uintptr_t)buf & 15) return fail_msg("xmap_ingest_line_masks: buffer not 16-byte aligned");
    if (size == 0) return 0;
    const long long nch = (size + 15) / 16;
    ingest_mask_kernel<<<blocks_of(nch), ING_BLOCK, 0, (cudaStream_t)stream>>>((const uint4 *)buf, (long long)size,
                                                                                masks, block_cnt);
    XMAP_LAUNCH_CHECK();
    return 0;
}

extern "C" int xmap_ingest_line_offsets(const uint16_t *masks, int64_t size, const int64_t *block_off, int64_t *offs,
                                        void *stream) {
    if (size <= 0) return 0;
    const long long nch = (size + 15) / 16;
    ingest_offset_kernel<<<blocks_of(nch), ING_BLOCK, 0, (cudaStream_t)stream>>>(masks, nch, block_off, offs);
    XMAP_LAUNCH_CHECK();
    return 0;
}

extern "C" int xmap_ingest_parse(const uint8_t *buf, const int64_t *offs, int64_t n_lines, const char *label_h,
                                 int32_t label_len, double ts_min, double ts_max, int64_t ld, uint8_t *status,
                                 double *rating, double *ts, uint64_t *uid_words, uint8_t *uid_len, uint64_t *iid_words,
                                 uint8_t *iid_len, void *stream) {
    if (label_len < 0 || label_len > 16) return fail_msg("xmap_ingest_parse: the domain label is longer than 16 bytes");
    if (n_lines <= 0) return 0;
    unsigned long long l0 = 0, l1 = 0;
    for (int k = 0; k < 16; ++k) {
        const unsigned long long c = k < label_len ? (uint8_t)label_h[k] : 0u;
        if (k < 8) l0 = (l0 << 8) | c;
        else l1 = (l1 << 8) | c;
    }
    const unsigned g = (unsigned)((n_lines + 32 * ING_WARPS - 1) / (32 * ING_WARPS));
    ingest_parse_kernel<<<g, ING_BLOCK, 0, (cudaStream_t)stream>>>(
        buf, offs, (long long)n_lines, l0, l1, label_len, ts_min, ts_max, (long long)ld, status, rating, ts,
        (unsigned long long *)uid_words, uid_len, (unsigned long long *)iid_words, iid_len);
    XMAP_LAUNCH_CHECK();
    return 0;
}

extern "C" int xmap_ingest_rank_flags(const uint64_t *words, int64_t ld, int32_t n_words, const int64_t *perm, int64_t n,
                                      int32_t *flag, void *stream) {
    if (n_words < 1 || n_words > ING_WORDS) return fail_msg("xmap_ingest_rank_flags: bad word count");
    if (n <= 0) return 0;
    ingest_rank_flags_kernel<<<blocks_of(n), ING_BLOCK, 0, (cudaStream_t)stream>>>(
        (const unsigned long long *)words, (long long)ld, n_words, perm, (long long)n, flag);
    XMAP_LAUNCH_CHECK();
    return 0;
}

extern "C" int xmap_ingest_rank_scatter(const int64_t *perm, const int32_t *flag, const int64_t *csum, int64_t n,
                                        int32_t *rank, int64_t *rep, void *stream) {
    if (n <= 0) return 0;
    ingest_rank_scatter_kernel<<<blocks_of(n), ING_BLOCK, 0, (cudaStream_t)stream>>>(perm, flag, csum, (long long)n,
                                                                                      rank, rep);
    XMAP_LAUNCH_CHECK();
    return 0;
}

extern "C" int xmap_ingest_first(const int32_t *user, const int32_t *item, const double *ts, const int64_t *order,
                                 const uint8_t *keep, int64_t n, double t_lo, double t_hi, int32_t *first_user,
                                 int32_t *pair_first, void *stream) {
    if (n <= 0) return 0;
    ingest_first_kernel<<<blocks_of(n), ING_BLOCK, 0, (cudaStream_t)stream>>>(user, item, ts, order, keep, (long long)n,
                                                                               t_lo, t_hi, first_user, pair_first);
    XMAP_LAUNCH_CHECK();
    return 0;
}

extern "C" int xmap_ingest_item_suffix(const uint64_t *iid_words, int64_t ld, const uint8_t *iid_len, const int64_t *rep,
                                       int32_t n_items, uint8_t *present, void *stream) {
    if (n_items <= 0) return 0;
    ingest_item_suffix_kernel<<<blocks_of(n_items), ING_BLOCK, 0, (cudaStream_t)stream>>>(
        (const unsigned long long *)iid_words, (long long)ld, iid_len, rep, n_items, present);
    XMAP_LAUNCH_CHECK();
    return 0;
}

extern "C" int xmap_ingest_item_codes(const uint64_t *iid_words, int64_t ld, const uint8_t *iid_len, const int64_t *rep,
                                      int32_t n_items, const int32_t *labels, int32_t n_labels, int32_t *prefix_new,
                                      uint8_t *dom_code, uint8_t *contains, bool *has_S, bool *has_T, void *stream) {
    if (n_labels < 0 || n_labels > 8) return fail_msg("xmap_ingest_item_codes: at most 8 domain labels");
    if (n_items <= 0) return 0;
    ingest_item_codes_kernel<<<blocks_of(n_items), ING_BLOCK, 0, (cudaStream_t)stream>>>(
        (const unsigned long long *)iid_words, (long long)ld, iid_len, rep, n_items, labels, n_labels, prefix_new,
        dom_code, contains, has_S, has_T);
    XMAP_LAUNCH_CHECK();
    return 0;
}

extern "C" int xmap_ingest_train_keys(const int32_t *user, const int32_t *item, const int8_t *grp, const int32_t *upos,
                                      const bool *has_S, const int32_t *srank, int64_t n, int64_t *key, void *stream) {
    if (n <= 0) return 0;
    ingest_train_keys_kernel<<<blocks_of(n), ING_BLOCK, 0, (cudaStream_t)stream>>>(user, item, grp, upos, has_S, srank,
                                                                                    (long long)n, key);
    XMAP_LAUNCH_CHECK();
    return 0;
}
