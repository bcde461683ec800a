// kj_mkfmi.cu -- index construction on the device: protein FASTA -> .fmi, byte for byte what kaiju-mkbwt + kaiju-mkfmi write.
//
// Text T: every sequence followed by its own terminator (code 0), N = residues + nseq rows.  Rows 0..nseq-1 are the terminators in
// input order (mkbwt.c:834-856 encodes the read order behind every sequence; terminators sort below all letters); the other
// M = N - nseq rows are the letter suffixes in lexicographic order, a terminator comparing by its sequence number.
//
// Suffix sort (prefix doubling): round 0 radix-sorts all letter suffixes on their first K letters packed into 64 bits (a terminator
// packs as 0 and ends the key).  Every suffix gets the rank nseq + (index of the first row of its group); only suffixes in groups of
// two or more stay in the tied list.  Round r >= 1 sorts the tied list on (group rank, rank of p + h), h = K << (r-1) -- except that
// when p + h reaches the terminator of p's sequence the second key is that terminator's rank, i.e. the sequence number (it never
// looks into the next sequence).  The radix sort, the scans and the compactions are written here (no CUB / Thrust).
//
// Assembly, also on the device: the BWT (row of a sequence-start suffix -> 0), the lexicographic rank of every sequence (= order of
// its start suffix; empty sequences first), the packed SA samples (suffixArray.c:195-226), the letter counts behind startLcode
// (compactfmi.c:109-151), the per-256-row FMIrecode (compactfmi.c:402-439) and the index1 / index2 tables (fmicommon.h:104-171).
#include <cuda_runtime.h>
#include <stdint.h>
#include <algorithm>
#include <cctype>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include "kj_host.h"

namespace {

#define MK_CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { kj_err() = std::string("kj_mkfmi: ") + #x + ": " + cudaGetErrorString(e_); return KJ_ERR_CUDA; } } while (0)

constexpr int SCAN_TILE = 2048;                    // 256 threads x 8 items
constexpr int RS_THREADS = 256, RS_IPT = 32;       // radix sort: 256 threads, 32 sub-tiles of 256 items
constexpr uint32_t RS_TILE = RS_THREADS * RS_IPT;

static inline int bits_needed(uint64_t k) { int i = 0; while (i < 64 && (k >> i)) ++i; return i; }     // suffixArray.c:58
static inline uint64_t cdiv(uint64_t a, uint64_t b) { return (a + b - 1) / b; }

// ------------------------------------------------------------------------------------------------ scans
__global__ void k_scan_tile(const uint32_t* __restrict__ in, uint32_t* __restrict__ out, uint32_t* __restrict__ bsum, uint64_t n) {
    __shared__ uint32_t s_w[8];
    const uint64_t base = (uint64_t)blockIdx.x * SCAN_TILE + threadIdx.x * 8ull;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t v[8], sum = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) { v[k] = base + k < n ? in[base + k] : 0u; sum += v[k]; }
    uint32_t x = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    if (lane == 31) s_w[warp] = x;
    __syncthreads();
    if (warp == 0) {
        uint32_t w = lane < 8 ? s_w[lane] : 0u;
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, w, o); if (lane >= o) w += y; }
        if (lane < 8) s_w[lane] = w;
    }
    __syncthreads();
    uint32_t pre = x - sum + (warp ? s_w[warp - 1] : 0u);
#pragma unroll
    for (int k = 0; k < 8; k++) if (base + k < n) { out[base + k] = pre; pre += v[k]; }
    if (bsum && threadIdx.x == 255) bsum[blockIdx.x] = s_w[7];
}
__global__ void k_scan_add(uint32_t* __restrict__ out, const uint32_t* __restrict__ add, uint64_t n) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] += add[i / SCAN_TILE];
}

struct Dev {
    cudaStream_t st = nullptr;
    uint32_t* scan_pool = nullptr; uint64_t scan_pool_n = 0;
    uint64_t* d_scalar = nullptr;                  // small D2H staging
    uint64_t sort_bytes = 0;
};

// exclusive scan of n uint32 (in != out); the scan of the tile sums recurses into the pool
static int scan_excl(Dev& D, const uint32_t* in, uint32_t* out, uint64_t n, uint32_t* pool) {
    if (n == 0) return KJ_OK;
    const uint64_t nb = cdiv(n, SCAN_TILE);
    if (nb == 1) { k_scan_tile<<<1, 256, 0, D.st>>>(in, out, nullptr, n); return cudaGetLastError() == cudaSuccess ? KJ_OK : KJ_ERR_CUDA; }
    uint32_t* bs = pool; uint32_t* bss = pool + nb;
    k_scan_tile<<<(unsigned)nb, 256, 0, D.st>>>(in, out, bs, n);
    int rc = scan_excl(D, bs, bss, nb, pool + 2 * nb); if (rc) return rc;
    k_scan_add<<<(unsigned)cdiv(n, 256), 256, 0, D.st>>>(out, bss, n);
    return cudaGetLastError() == cudaSuccess ? KJ_OK : KJ_ERR_CUDA;
}
static uint64_t scan_pool_size(uint64_t n) { uint64_t s = 0; while (n > SCAN_TILE) { n = cdiv(n, SCAN_TILE); s += 2 * n; } return s + 16; }

__global__ void k_total(const uint32_t* flags, const uint32_t* ex, uint64_t n, uint64_t* out) { *out = (uint64_t)ex[n - 1] + flags[n - 1]; }
// exclusive scan + the total on the host (one small copy; the callers need the count to size the next launch)
static int scan_count(Dev& D, const uint32_t* flags, uint32_t* ex, uint64_t n, uint64_t& total) {
    total = 0; if (n == 0) return KJ_OK;
    if (scan_excl(D, flags, ex, n, D.scan_pool)) { kj_err() = "kj_mkfmi: scan launch failed"; return KJ_ERR_CUDA; }
    k_total<<<1, 1, 0, D.st>>>(flags, ex, n, D.d_scalar);
    MK_CK(cudaMemcpyAsync(&total, D.d_scalar, 8, cudaMemcpyDeviceToHost, D.st));
    MK_CK(cudaStreamSynchronize(D.st));
    return KJ_OK;
}

// ------------------------------------------------------------------------------------------------ LSD radix sort (uint64 key, uint32 value), stable
__global__ void k_rs_hist(const uint64_t* __restrict__ key, uint64_t n, int shift, uint32_t* __restrict__ hist, uint32_t nblk) {
    __shared__ uint32_t s_h[256];
    s_h[threadIdx.x] = 0;
    __syncthreads();
    const uint64_t base = (uint64_t)blockIdx.x * RS_TILE;
    for (int r = 0; r < RS_IPT; r++) {
        const uint64_t i = base + (uint64_t)r * RS_THREADS + threadIdx.x;
        if (i < n) atomicAdd(&s_h[(key[i] >> shift) & 255u], 1u);
    }
    __syncthreads();
    hist[(uint64_t)threadIdx.x * nblk + blockIdx.x] = s_h[threadIdx.x];
}
// each sub-tile of 256 items is ranked warp by warp (__match_any_sync) so that equal digits keep their input order
__global__ void k_rs_scatter(const uint64_t* __restrict__ key, const uint32_t* __restrict__ val, uint64_t n, int shift,
                             const uint32_t* __restrict__ off, uint32_t nblk, uint64_t* __restrict__ key_out, uint32_t* __restrict__ val_out) {
    __shared__ uint32_t s_base[256];
    __shared__ uint32_t s_w[8][256];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    s_base[threadIdx.x] = off[(uint64_t)threadIdx.x * nblk + blockIdx.x];
    for (int w = 0; w < 8; w++) s_w[w][threadIdx.x] = 0;
    __syncthreads();
    const uint64_t base = (uint64_t)blockIdx.x * RS_TILE;
    const uint32_t lt = (1u << lane) - 1u;
    for (int r = 0; r < RS_IPT; r++) {
        if (base + (uint64_t)r * RS_THREADS >= n) break;                       // uniform over the block
        const uint64_t i = base + (uint64_t)r * RS_THREADS + threadIdx.x;
        const bool ok = i < n;
        const uint64_t k = ok ? key[i] : 0; const uint32_t v = ok ? val[i] : 0;
        const uint32_t d = ok ? (uint32_t)((k >> shift) & 255u) : 256u;
        const uint32_t peers = __match_any_sync(0xffffffffu, d);
        const uint32_t rank = __popc(peers & lt);
        if (ok && rank == 0) s_w[warp][d] = __popc(peers);
        __syncthreads();
        {   // digit threadIdx.x: offsets of the 8 warps' runs, then advance the block's base for the next sub-tile
            uint32_t run = s_base[threadIdx.x];
#pragma unroll
            for (int w = 0; w < 8; w++) { const uint32_t c = s_w[w][threadIdx.x]; s_w[w][threadIdx.x] = run; run += c; }
            s_base[threadIdx.x] = run;
        }
        __syncthreads();
        if (ok) { const uint32_t pos = s_w[warp][d] + rank; key_out[pos] = k; val_out[pos] = v; }
        __syncthreads();
#pragma unroll
        for (int w = 0; w < 8; w++) s_w[w][threadIdx.x] = 0;
        __syncthreads();
    }
}

struct SortBufs { uint64_t* k[2]; uint32_t* v[2]; uint32_t* hist; uint32_t* off; };

// sorts (k[0], v[0]) on the low `bits` bits of the key; returns which buffer pair holds the result
static int radix_sort(Dev& D, SortBufs& B, uint64_t n, int bits, int& which) {
    which = 0;
    if (n <= 1) return KJ_OK;
    const uint32_t nblk = (uint32_t)cdiv(n, RS_TILE);
    for (int shift = 0; shift < bits; shift += 8) {
        k_rs_hist<<<nblk, RS_THREADS, 0, D.st>>>(B.k[which], n, shift, B.hist, nblk);
        if (scan_excl(D, B.hist, B.off, (uint64_t)nblk * 256, D.scan_pool)) { kj_err() = "kj_mkfmi: scan launch failed"; return KJ_ERR_CUDA; }
        k_rs_scatter<<<nblk, RS_THREADS, 0, D.st>>>(B.k[which], B.v[which], n, shift, B.off, nblk, B.k[which ^ 1], B.v[which ^ 1]);
        MK_CK(cudaGetLastError());
        which ^= 1;
        D.sort_bytes += n * 8 + 2 * n * 12 + (uint64_t)nblk * 256 * 4 * 4;   // hist read of keys, scatter read + write, histogram + scan
    }
    return KJ_OK;
}

// ------------------------------------------------------------------------------------------------ suffix sort kernels
// sequence of text position p: the last s with start[s] <= p (start[nseq] = N)
__device__ __forceinline__ uint32_t seq_of(const uint32_t* __restrict__ start, uint32_t nseq, uint64_t p) {
    uint32_t lo = 0, hi = nseq - 1;
    while (lo < hi) { const uint32_t mid = (uint32_t)(((uint64_t)lo + hi + 1) >> 1); if (start[mid] <= p) lo = mid; else hi = mid - 1; }
    return lo;
}
__global__ void k_letter_flags(const uint8_t* __restrict__ T, uint64_t N, uint32_t* __restrict__ f) {
    const uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < N) f[p] = T[p] != 0;
}
// position list of the letters + their round-0 keys: K letters of `sb` bits each, most significant first, 0 from the terminator on
__global__ void k_init_keys(const uint8_t* __restrict__ T, uint64_t N, const uint32_t* __restrict__ f, const uint32_t* __restrict__ ex,
                            int K, int sb, uint64_t* __restrict__ key, uint32_t* __restrict__ pos) {
    const uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= N || !f[p]) return;
    uint64_t k = 0; bool end = false;
    for (int j = 0; j < K; j++) {
        uint32_t c = 0;
        if (!end) { c = p + j < N ? T[p + j] : 0; if (c == 0) end = true; }
        k = (k << sb) | c;
    }
    key[ex[p]] = k; pos[ex[p]] = (uint32_t)p;
}
// heads of the groups of equal keys in a sorted list, the tied flags come after the scan
__global__ void k_heads(const uint64_t* __restrict__ key, uint64_t n, uint32_t* __restrict__ h) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n) h[j] = (j == 0 || key[j] != key[j - 1]) ? 1u : 0u;
}
// gid = ex[j] + h[j] - 1; gstart[gid] = row index (in SA order) of the group's first element
__global__ void k_group_start(const uint32_t* __restrict__ h, const uint32_t* __restrict__ ex, const uint32_t* __restrict__ idx, uint64_t n, uint32_t* __restrict__ gstart) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n && h[j]) gstart[ex[j]] = idx ? idx[j] : (uint32_t)j;
}
// writes the sorted positions back into the SA, the new ranks, and the tied flags (groups of >= 2)
__global__ void k_apply(const uint32_t* __restrict__ h, const uint32_t* __restrict__ ex, const uint32_t* __restrict__ gstart, const uint32_t* __restrict__ idx,
                        const uint32_t* __restrict__ psorted, uint64_t n, uint32_t nseq, uint32_t* __restrict__ sa, uint32_t* __restrict__ rank, uint32_t* __restrict__ tied) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const uint32_t p = psorted[j];
    const uint32_t row = idx ? idx[j] : (uint32_t)j;
    sa[row] = p;
    rank[p] = nseq + gstart[ex[j] + h[j] - 1];
    tied[j] = !(h[j] && (j + 1 == n || h[j + 1]));
}
__global__ void k_compact_idx(const uint32_t* __restrict__ tied, const uint32_t* __restrict__ ex, const uint32_t* __restrict__ idx, uint64_t n, uint32_t* __restrict__ out) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n && tied[j]) out[ex[j]] = idx ? idx[j] : (uint32_t)j;
}
// round keys of the tied list: (group rank | rank at p + h, or the terminator's rank = sequence number once p + h reaches it)
__global__ void k_round_keys(const uint32_t* __restrict__ idx, uint64_t n, const uint32_t* __restrict__ sa, const uint32_t* __restrict__ rank,
                             const uint32_t* __restrict__ start, uint32_t nseq, uint64_t h, int rbits, uint64_t* __restrict__ key, uint32_t* __restrict__ pos) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const uint32_t p = sa[idx[j]];
    const uint32_t s = seq_of(start, nseq, p);
    const uint64_t term = (uint64_t)start[s + 1] - 1;
    const uint32_t r2 = (uint64_t)p + h >= term ? s : rank[p + h];
    key[j] = ((uint64_t)(rank[p] - nseq) << rbits) | r2;
    pos[j] = p;
}

// ------------------------------------------------------------------------------------------------ assembly kernels
__global__ void k_bwt(const uint8_t* __restrict__ T, const uint32_t* __restrict__ sa, const uint32_t* __restrict__ start, uint32_t nseq, uint64_t N, uint8_t* __restrict__ bwt) {
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= N) return;
    const uint64_t p = r < nseq ? (uint64_t)start[r + 1] - 1 : sa[r - nseq];        // terminator row r: the terminator of sequence r
    bwt[r] = p ? T[p - 1] : 0;
}
__global__ void k_start_flags(const uint8_t* __restrict__ bwt, uint32_t nseq, uint64_t M, uint32_t* __restrict__ f) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < M) f[i] = bwt[nseq + i] == 0;
}
__global__ void k_empty_flags(const uint32_t* __restrict__ start, uint32_t nseq, uint32_t* __restrict__ f) {
    const uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s < nseq) f[s] = start[s + 1] - start[s] == 1;
}
// lexicographic rank of every sequence (mkbwt.c:700-728: sequence text, then its terminator) and its inverse, seqTermOrder
__global__ void k_lex_empty(const uint32_t* __restrict__ fe, const uint32_t* __restrict__ exe, uint32_t nseq, uint32_t* __restrict__ lex, uint32_t* __restrict__ order) {
    const uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s < nseq && fe[s]) { lex[s] = exe[s]; order[exe[s]] = (uint32_t)s; }
}
__global__ void k_lex_letters(const uint32_t* __restrict__ fs, const uint32_t* __restrict__ exs, const uint32_t* __restrict__ sa, const uint32_t* __restrict__ start,
                              uint32_t nseq, uint64_t M, uint32_t n_empty, uint32_t* __restrict__ lex, uint32_t* __restrict__ order) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M || !fs[i]) return;
    const uint32_t s = seq_of(start, nseq, sa[i]);
    const uint32_t r = n_empty + exs[i];
    lex[s] = r; order[r] = s;
}
// SA sample q = row ((((nseq-1) >> e) + 1 + q) << e): (lex rank << pbits) + position, big-endian in nbytes (suffixArray.c:40-53)
__global__ void k_samples(const uint32_t* __restrict__ sa, const uint32_t* __restrict__ start, const uint32_t* __restrict__ lex, uint32_t nseq, int e,
                          uint64_t nsamp, int pbits, int nbytes, uint8_t* __restrict__ out) {
    const uint64_t q = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nsamp) return;
    const uint64_t row = ((((uint64_t)nseq - 1) >> e) + 1 + q) << e;
    const uint32_t p = sa[row - nseq];
    const uint32_t s = seq_of(start, nseq, p);
    uint64_t v = ((uint64_t)lex[s] << pbits) + (p - start[s]);
    for (int b = nbytes - 1; b >= 0; b--) { out[q * nbytes + b] = (uint8_t)v; v >>= 8; }
}
// letter counts of every 256-row block: cnt[a * nblk + b]
__global__ void k_block_counts(const uint8_t* __restrict__ bwt, uint64_t N, int alen, uint64_t nblk, uint32_t* __restrict__ cnt) {
    __shared__ uint32_t s_c[32];
    if (threadIdx.x < 32) s_c[threadIdx.x] = 0;
    __syncthreads();
    const uint64_t r = (uint64_t)blockIdx.x * 256 + threadIdx.x;
    if (r < N) atomicAdd(&s_c[bwt[r]], 1u);
    __syncthreads();
    if (threadIdx.x < alen) cnt[(uint64_t)threadIdx.x * nblk + blockIdx.x] = s_c[threadIdx.x];
}
__global__ void k_letter_totals(const uint32_t* __restrict__ cnt, const uint32_t* __restrict__ cum, uint64_t nblk, int alen, uint64_t* __restrict__ tot) {
    const int a = threadIdx.x;
    if (a < alen) tot[a] = (uint64_t)cum[(uint64_t)a * nblk + nblk - 1] + cnt[(uint64_t)a * nblk + nblk - 1];
}
// FMIrecode (compactfmi.c:402-439): in each 256-row block the first half stores the count of its letter before it in the block, the
// second half the count after it, both capped at the letter's code range (startLcode)
__global__ void k_recode(const uint8_t* __restrict__ bwt, uint64_t N, const int* __restrict__ startL, uint8_t* __restrict__ out) {
    __shared__ uint32_t s_w[8][32];
    __shared__ int s_L[33];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x < 33) s_L[threadIdx.x] = startL[threadIdx.x];
    s_w[warp][lane] = 0;
    __syncthreads();
    const uint64_t r = (uint64_t)blockIdx.x * 256 + threadIdx.x;
    const bool ok = r < N;
    const uint32_t c = ok ? bwt[r] : 32u;
    const uint32_t peers = __match_any_sync(0xffffffffu, c);
    const uint32_t rank = __popc(peers & ((1u << lane) - 1u));
    if (ok && rank == 0) s_w[warp][c] = __popc(peers);
    __syncthreads();
    if (!ok) return;
    uint32_t before = rank, total = 0;
    for (int w = 0; w < 8; w++) { const uint32_t k = s_w[w][c]; if (w < warp) before += k; total += k; }
    int n = threadIdx.x < 128 ? (int)before : (int)(total - before) - 1;
    const int mx = s_L[c + 1] - s_L[c] - 1;
    if (n > mx) n = mx;
    out[r] = (uint8_t)(s_L[c] + n);
}
// index1 [N1][alen] (fmicommon.h:127-130, 162-165) and index2 [N2][alen] (132-136, 155-157), from the per-block cumulative counts
__global__ void k_index_tables(const uint32_t* __restrict__ cum, const uint64_t* __restrict__ tot, uint64_t nblk, int alen, uint64_t N,
                               int64_t N1, int64_t N2, int64_t* __restrict__ index1, uint16_t* __restrict__ index2) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t last1 = (N - 1) >> 16;                       // the checkpoint-1 row of the last position
    if (t < (uint64_t)N2 * alen) {
        const uint64_t R2 = t / alen; const int a = (int)(t % alen);
        uint64_t v;
        if ((int64_t)R2 == N2 - 1) v = tot[a] - cum[(uint64_t)a * nblk + (last1 << 8)];
        else v = (uint64_t)cum[(uint64_t)a * nblk + R2] - cum[(uint64_t)a * nblk + ((R2 >> 8) << 8)];
        index2[t] = (uint16_t)v;
    }
    if (t < (uint64_t)N1 * alen) {
        const uint64_t R1 = t / alen; const int a = (int)(t % alen);
        uint64_t Ca = 0; for (int b = 0; b < a; b++) Ca += tot[b];
        index1[t] = (int64_t)R1 == N1 - 1 ? (int64_t)Ca : (int64_t)cum[(uint64_t)a * nblk + (R1 << 8)] + (a ? (int64_t)Ca : 0);
    }
}

// ------------------------------------------------------------------------------------------------ host: FASTA (readFasta.c:99-163)
struct Faa {
    std::vector<uint8_t> T;                        // residues with a 0 after every sequence
    std::vector<uint32_t> start;                   // [nseq + 1]
    std::vector<std::string> ids;                  // cut at the first blank, at most 255 bytes (suffixArray.c:232-240)
    uint64_t maxlen = 0;
};
struct ByteIn {
    FILE* fp; std::vector<uint8_t> buf; size_t pos = 0, len = 0;
    explicit ByteIn(FILE* f) : fp(f), buf(1 << 22) {}
    int get() { if (pos == len) { len = fread(buf.data(), 1, buf.size(), fp); pos = 0; if (!len) return EOF; } return buf[pos++]; }
};

static int parse_faa(const char* path, const std::string& letters, Faa& F) {
    FILE* fp = fopen(path, "rb");
    if (!fp) { kj_err() = std::string("kj_mkfmi: could not open ") + path; return KJ_ERR_IO; }
    // translation_table (sequence.c:68-97): letters of the alphabet (either case) -> 1.., other letters -> the last letter, '*' -> 0
    int8_t tr[256];
    const int nl = (int)letters.size();
    for (int i = 0; i < 256; i++) tr[i] = (i < 128 && isalpha(i)) ? (int8_t)nl : (int8_t)-1;
    for (int i = 0; i < nl; i++) { tr[toupper((unsigned char)letters[i])] = (int8_t)(i + 1); tr[tolower((unsigned char)letters[i])] = (int8_t)(i + 1); }
    tr[0] = 0; tr[(unsigned char)'*'] = 0;
    ByteIn in(fp);
    int c;
    do c = in.get(); while (c != '>' && c != EOF);
    int rc = KJ_OK;
    std::string line;
    while (c != EOF) {
        // id line: fgets of at most 999 bytes, the rest of a longer line is dropped, the last byte read is cut (read_id, 49-81)
        line.clear(); int d = 0;
        while ((int)line.size() < 999) { d = in.get(); if (d == EOF) break; line.push_back((char)d); if (d == '\n') break; }
        if (line.empty()) { kj_err() = "kj_mkfmi: the input ends inside an id line"; rc = KJ_ERR_IO; break; }
        if (line.back() != '\n') {
            do d = in.get(); while (d != '\n' && d != EOF);
            if (d == EOF) { kj_err() = "kj_mkfmi: the input ends inside an id line"; rc = KJ_ERR_IO; break; }
        }
        line.pop_back();
        size_t cut = 0; while (cut < line.size() && line[cut] != '\0' && line[cut] != ' ' && line[cut] != '\t') ++cut;
        F.ids.push_back(line.substr(0, cut < 255 ? cut : 255));
        F.start.push_back((uint32_t)F.T.size());
        const uint64_t s0 = F.T.size();
        int last = 0;
        c = in.get();
        while (c != EOF) {
            if (c == '>' && last == '\n') break;           // a record ends at "\n>"; a '>' anywhere else is skipped like any non-letter
            const int8_t t = tr[c];
            if (t > 0) F.T.push_back((uint8_t)t);
            else if (t == 0) { kj_err() = "kj_mkfmi: sequence " + F.ids.back() + " contains the terminator character '*' (or a NUL byte); kaiju-mkbwt reads it as a sequence end and writes an inconsistent BWT"; rc = KJ_ERR_UNSUPPORTED; break; }
            last = c; c = in.get();
        }
        if (rc) break;
        const uint64_t len = F.T.size() - s0;
        if (len > F.maxlen) F.maxlen = len;
        F.T.push_back(0);
        if (F.T.size() >= (1ull << 32)) { kj_err() = "kj_mkfmi: the index would have 2^32 rows or more (out of core construction is not supported)"; rc = KJ_ERR_UNSUPPORTED; break; }
    }
    fclose(fp);
    if (rc) return rc;
    if (F.ids.empty()) { kj_err() = std::string("kj_mkfmi: no sequence in ") + path; return KJ_ERR_UNSUPPORTED; }
    F.start.push_back((uint32_t)F.T.size());
    return KJ_OK;
}

// find_startLcode (compactfmi.c:109-151), the double arithmetic included
static void start_lcode(const uint64_t* count, int alen, int* startL) {
    uint64_t tot = 0; for (int a = 0; a < alen; a++) tot += count[a];
    int maxN[32] = {0}, sum = 0, mx = 0;
    for (int a = 0; a < alen; a++) {
        maxN[a] = (int)(256 * ((double)count[a] / tot));
        if (maxN[a] < 2) maxN[a] = 2;
        if (maxN[a] > maxN[mx]) mx = a;
        sum += maxN[a];
    }
    if (sum < 256) maxN[mx] += 256 - sum;
    while (sum > 256) {
        int mn = 0;
        for (int a = 1; a < alen; a++) { if (maxN[mn] <= 2) mn = a; if (maxN[a] > 2 && maxN[a] < maxN[mn]) mn = a; }
        maxN[mn] -= 1; sum -= 1;
    }
    startL[0] = 0; startL[alen] = 256;
    for (int a = 0; a < alen; a++) startL[a + 1] = startL[a] + maxN[a];
}

struct Out {
    std::vector<uint8_t> bwt, recoded, samples; std::vector<uint32_t> order;
    std::vector<int64_t> index1; std::vector<uint16_t> index2; int startL[33] = {0};
    int64_t N1 = 0, N2 = 0; uint64_t nsamp = 0;
};

struct Writer {
    FILE* fp; bool ok = true;
    explicit Writer(FILE* f) : fp(f) {}
    template <class T> void put(T v) { if (fwrite(&v, sizeof v, 1, fp) != 1) ok = false; }
    void bytes(const void* p, size_t n) { if (n && fwrite(p, 1, n, fp) != n) ok = false; }
};

struct SaHeader { int64_t len, ncheck; int32_t e, nbytes, sbits, pbits; int64_t mask, check; };

static void write_sa_header(Writer& w, const SaHeader& h, const Faa& F, const Out& O) {          // suffixArray.c:261-277
    const int32_t nseq = (int32_t)F.ids.size();
    w.put(h.len); w.put(h.ncheck); w.put(h.e); w.put(h.nbytes); w.put(h.sbits); w.put(h.pbits); w.put(h.mask); w.put(h.check); w.put(nseq);
    for (int32_t i = 0; i < nseq; i++) { const std::string& id = F.ids[O.order[i]]; w.put((uint8_t)id.size()); w.bytes(id.data(), id.size()); }
    for (int32_t i = 0; i < nseq; i++) w.put((int32_t)O.order[i]);
    for (int32_t i = 0; i < nseq; i++) { const uint32_t s = O.order[i]; w.put((int64_t)(F.start[s + 1] - F.start[s] - 1)); }
}

static int write_files(const char* prefix, const Faa& F, const Out& O, const std::string& alphabet, int e, bool bwt_sa) {
    const int64_t N = (int64_t)F.T.size(); const int32_t nseq = (int32_t)F.ids.size(), alen = (int32_t)alphabet.size();
    SaHeader h;
    h.len = N; h.ncheck = (N >> e) - ((int64_t)nseq >> e); h.e = e;
    h.sbits = bits_needed((uint64_t)nseq); h.pbits = bits_needed(F.maxlen); h.nbytes = (7 + h.sbits + h.pbits) / 8;
    h.mask = (int64_t)(int32_t)(uint32_t)((1ull << h.pbits) - 1); h.check = (int64_t)(int32_t)(uint32_t)((1ull << e) - 1);   // int arithmetic in the reference
    auto open = [&](const char* ext, FILE*& fp) { fp = fopen((std::string(prefix) + ext).c_str(), "wb"); if (!fp) kj_err() = std::string("kj_mkfmi: could not create ") + prefix + ext; return fp != nullptr; };
    auto bwt_header = [&](Writer& w) { w.put(N); w.put(nseq); w.put(alen); w.bytes(alphabet.data(), alen); };        // bwt.c:40-45
    FILE* fp;
    if (bwt_sa) {
        if (!open(".bwt", fp)) return KJ_ERR_IO;
        Writer w(fp); bwt_header(w); w.bytes(O.bwt.data(), N);
        if (fclose(fp) != 0 || !w.ok) { kj_err() = "kj_mkfmi: write error on .bwt"; return KJ_ERR_IO; }
        if (!open(".sa", fp)) return KJ_ERR_IO;
        Writer s(fp); write_sa_header(s, h, F, O); s.bytes(O.samples.data(), O.nsamp * h.nbytes);
        if (fclose(fp) != 0 || !s.ok) { kj_err() = "kj_mkfmi: write error on .sa"; return KJ_ERR_IO; }
    }
    // mkfmi.c:63-78: BWT header, suffix-array header + its first ncheck samples (one fewer than mkbwt wrote when nseq is a multiple of
    // 2^e, one more -- zero -- when bwtlen is and nseq is not), then the FM index
    if (!open(".fmi", fp)) return KJ_ERR_IO;
    Writer w(fp); bwt_header(w); write_sa_header(w, h, F, O);
    const uint64_t keep = std::min<uint64_t>((uint64_t)h.ncheck, O.nsamp);
    w.bytes(O.samples.data(), keep * h.nbytes);
    if ((uint64_t)h.ncheck > keep) { std::vector<uint8_t> z(((uint64_t)h.ncheck - keep) * h.nbytes, 0); w.bytes(z.data(), z.size()); }
    w.put(alen); w.put(N); w.put((int32_t)O.N1); w.put((int32_t)O.N2);                                             // fmicommon.h:175-184
    w.bytes(O.recoded.data(), N);
    w.bytes(O.index1.data(), O.index1.size() * 8); w.bytes(O.index2.data(), O.index2.size() * 2);
    w.bytes(O.startL, (alen + 1) * sizeof(int));
    if (fclose(fp) != 0 || !w.ok) { kj_err() = "kj_mkfmi: write error on .fmi"; return KJ_ERR_IO; }
    return KJ_OK;
}

struct DevMem {
    std::vector<void*> ptrs;
    ~DevMem() { for (void* p : ptrs) cudaFree(p); }
    template <class T> int alloc(T*& p, uint64_t n) {
        void* q = nullptr;
        if (cudaMalloc(&q, n ? n * sizeof(T) : 1) != cudaSuccess) { cudaGetLastError(); kj_err() = "kj_mkfmi: cudaMalloc failed"; return KJ_ERR_NOMEM; }
        ptrs.push_back(q); p = (T*)q; return KJ_OK;
    }
    void release(void* p) { for (auto& q : ptrs) if (q == p) { cudaFree(q); q = nullptr; } }
};

static inline unsigned grid(uint64_t n, unsigned b = 256) { return (unsigned)std::max<uint64_t>(1, cdiv(n, b)); }
using clk = std::chrono::steady_clock;
static inline double ms_since(clk::time_point t) { return std::chrono::duration<double, std::milli>(clk::now() - t).count(); }

static int build(const Faa& F, int alen, int e, Out& O, kj_mkfmi_stats& S, Dev& D) {
    const uint64_t N = F.T.size(); const uint32_t nseq = (uint32_t)F.ids.size(); const uint64_t M = N - nseq;
    const uint64_t scanN = scan_pool_size(std::max<uint64_t>(N, (uint64_t)cdiv(std::max<uint64_t>(M, 1), RS_TILE) * 256));
    // memory estimate (bytes): text 1 + rank 4 per row; per letter suffix: SA 4, sort keys 2 x 8, values 2 x 4, scratch 3 x 4
    const uint64_t need = N * 5 + M * (4 + 16 + 8 + 12) + scanN * 4 + cdiv(M, RS_TILE) * 256 * 8 + (1 << 20);
    size_t fre = 0, totm = 0;
    MK_CK(cudaMemGetInfo(&fre, &totm));
    if (need > fre) { kj_err() = "kj_mkfmi: the construction needs about " + std::to_string(need >> 20) + " MiB of device memory, " + std::to_string(fre >> 20) + " MiB are free"; return KJ_ERR_NOMEM; }
    auto t0 = clk::now();
    DevMem mem; int rc;
    uint8_t* dT; uint32_t *dstart, *drank, *dsa, *s1, *s2, *s3; SortBufs B;
    if ((rc = mem.alloc(dT, N)) || (rc = mem.alloc(dstart, nseq + 1)) || (rc = mem.alloc(drank, N)) || (rc = mem.alloc(dsa, M)) ||
        (rc = mem.alloc(s1, std::max<uint64_t>(N, M))) || (rc = mem.alloc(s2, std::max<uint64_t>(N, M))) || (rc = mem.alloc(s3, M)) ||
        (rc = mem.alloc(B.k[0], M)) || (rc = mem.alloc(B.k[1], M)) || (rc = mem.alloc(B.v[0], M)) || (rc = mem.alloc(B.v[1], M)) ||
        (rc = mem.alloc(B.hist, cdiv(M, RS_TILE) * 256)) || (rc = mem.alloc(B.off, cdiv(M, RS_TILE) * 256)) ||
        (rc = mem.alloc(D.scan_pool, scanN)) || (rc = mem.alloc(D.d_scalar, 64))) return rc;
    MK_CK(cudaMemcpyAsync(dT, F.T.data(), N, cudaMemcpyHostToDevice, D.st));
    MK_CK(cudaMemcpyAsync(dstart, F.start.data(), (nseq + 1) * 4ull, cudaMemcpyHostToDevice, D.st));
    MK_CK(cudaStreamSynchronize(D.st));
    S.upload_ms = ms_since(t0);

    // ---- suffix sort
    t0 = clk::now();
    const int sb = bits_needed((uint64_t)alen - 1), K = 64 / sb;
    uint64_t cnt = 0;
    k_letter_flags<<<grid(N), 256, 0, D.st>>>(dT, N, s1);
    if ((rc = scan_count(D, s1, s2, N, cnt))) return rc;
    k_init_keys<<<grid(N), 256, 0, D.st>>>(dT, N, s1, s2, K, sb, B.k[0], B.v[0]);
    MK_CK(cudaGetLastError());
    const int rbits = bits_needed(N - 1), hbits = bits_needed(M ? M - 1 : 0);
    // per round: heads -> hb, their scan -> s2, group starts + tied flags -> the spare key buffer, the tied scan -> the spare value buffer;
    // the next tied list is compacted into hb (dead by then), so the tied list and the head flags alternate between s1 and s3
    uint32_t* idx = nullptr;                       // tied rows (SA order); nullptr in round 0 = all rows
    uint64_t n = M; int round = 0; uint64_t h = (uint64_t)K;
    while (n) {
        if (round >= KJ_MKFMI_MAX_ROUNDS) { kj_err() = "kj_mkfmi: the suffix sort did not converge"; return KJ_ERR_CUDA; }
        if (round > 0) {
            k_round_keys<<<grid(n), 256, 0, D.st>>>(idx, n, dsa, drank, dstart, nseq, h, rbits, B.k[0], B.v[0]);
            MK_CK(cudaGetLastError());
            h <<= 1;
        }
        int which = 0;
        if ((rc = radix_sort(D, B, n, round == 0 ? K * sb : hbits + rbits, which))) return rc;
        S.round_items[round] = n;
        // group heads -> group starts -> SA, ranks, tied flags -> the next tied list
        uint64_t ngroups = 0, ntied = 0;
        uint32_t* hb = (idx == s1) ? s3 : s1;
        k_heads<<<grid(n), 256, 0, D.st>>>(B.k[which], n, hb);
        if ((rc = scan_count(D, hb, s2, n, ngroups))) return rc;
        uint32_t* gstart = (uint32_t*)B.k[which ^ 1];            // the spare key buffer: 8 bytes per item = group starts + tied flags
        uint32_t* tied = gstart + n;
        k_group_start<<<grid(n), 256, 0, D.st>>>(hb, s2, idx, n, gstart);
        k_apply<<<grid(n), 256, 0, D.st>>>(hb, s2, gstart, idx, B.v[which], n, nseq, dsa, drank, tied);
        MK_CK(cudaGetLastError());
        uint32_t* tex = B.v[which ^ 1];
        if ((rc = scan_count(D, tied, tex, n, ntied))) return rc;
        k_compact_idx<<<grid(n), 256, 0, D.st>>>(tied, tex, idx, n, hb);
        MK_CK(cudaGetLastError());
        idx = hb; n = ntied; round++;
    }
    MK_CK(cudaStreamSynchronize(D.st));
    S.sort_rounds = round; S.sort_bytes = D.sort_bytes;
    S.sort_ms = ms_since(t0);

    // ---- assembly
    t0 = clk::now();
    mem.release(B.k[0]); mem.release(B.k[1]); mem.release(B.v[1]); mem.release(drank);
    uint8_t *dbwt, *drec; uint32_t *dlex, *dorder, *dcnt, *dcum; uint64_t* dtot; int* dL; int64_t* di1; uint16_t* di2; uint8_t* dsamp;
    const uint64_t nblk = cdiv(N, 256);
    O.N1 = (int64_t)((N - 1) >> 16) + 2; if (((uint64_t)O.N1 << 16) == N) O.N1 -= 1;                   // fmicommon.h:88-91, as written
    O.N2 = (int64_t)((N - 1) >> 8) + 2;  if (((uint64_t)O.N1 << 8) == N) O.N2 -= 1;
    O.nsamp = ((N - 1) >> e) - (((uint64_t)nseq - 1) >> e);
    const int pbits = bits_needed(F.maxlen), nbytes = (7 + bits_needed(nseq) + pbits) / 8;
    if ((rc = mem.alloc(dbwt, N)) || (rc = mem.alloc(drec, N)) || (rc = mem.alloc(dlex, nseq)) || (rc = mem.alloc(dorder, nseq)) ||
        (rc = mem.alloc(dcnt, nblk * alen)) || (rc = mem.alloc(dcum, nblk * alen)) || (rc = mem.alloc(dtot, 32)) || (rc = mem.alloc(dL, 33)) ||
        (rc = mem.alloc(di1, O.N1 * alen)) || (rc = mem.alloc(di2, O.N2 * alen)) || (rc = mem.alloc(dsamp, O.nsamp * nbytes))) return rc;
    k_bwt<<<grid(N), 256, 0, D.st>>>(dT, dsa, dstart, nseq, N, dbwt);
    uint64_t nstart = 0, nempty = 0;
    k_start_flags<<<grid(M), 256, 0, D.st>>>(dbwt, nseq, M, s1);
    if ((rc = scan_count(D, s1, s2, M, nstart))) return rc;
    uint32_t *fe, *exe;                                          // empty-sequence flags and their scan (nseq may exceed M)
    if ((rc = mem.alloc(fe, nseq)) || (rc = mem.alloc(exe, nseq))) return rc;
    k_empty_flags<<<grid(nseq), 256, 0, D.st>>>(dstart, nseq, fe);
    if ((rc = scan_count(D, fe, exe, nseq, nempty))) return rc;
    if (nstart + nempty != nseq) { kj_err() = "kj_mkfmi: internal error: sequence starts do not add up"; return KJ_ERR_CUDA; }
    k_lex_empty<<<grid(nseq), 256, 0, D.st>>>(fe, exe, nseq, dlex, dorder);
    k_lex_letters<<<grid(M), 256, 0, D.st>>>(s1, s2, dsa, dstart, nseq, M, (uint32_t)nempty, dlex, dorder);
    if (O.nsamp) k_samples<<<grid(O.nsamp), 256, 0, D.st>>>(dsa, dstart, dlex, nseq, e, O.nsamp, pbits, nbytes, dsamp);
    k_block_counts<<<(unsigned)nblk, 256, 0, D.st>>>(dbwt, N, alen, nblk, dcnt);
    MK_CK(cudaGetLastError());
    for (int a = 0; a < alen; a++)
        if (scan_excl(D, dcnt + (uint64_t)a * nblk, dcum + (uint64_t)a * nblk, nblk, D.scan_pool)) { kj_err() = "kj_mkfmi: scan launch failed"; return KJ_ERR_CUDA; }
    k_letter_totals<<<1, 32, 0, D.st>>>(dcnt, dcum, nblk, alen, dtot);
    uint64_t tot[32] = {0};
    MK_CK(cudaMemcpyAsync(tot, dtot, alen * 8, cudaMemcpyDeviceToHost, D.st));
    MK_CK(cudaStreamSynchronize(D.st));
    start_lcode(tot, alen, O.startL);
    MK_CK(cudaMemcpyAsync(dL, O.startL, 33 * sizeof(int), cudaMemcpyHostToDevice, D.st));
    k_recode<<<(unsigned)nblk, 256, 0, D.st>>>(dbwt, N, dL, drec);
    k_index_tables<<<grid((uint64_t)std::max(O.N1, O.N2) * alen), 256, 0, D.st>>>(dcum, dtot, nblk, alen, N, O.N1, O.N2, di1, di2);
    MK_CK(cudaGetLastError());
    O.bwt.resize(N); O.recoded.resize(N); O.order.resize(nseq); O.index1.resize(O.N1 * alen); O.index2.resize(O.N2 * alen); O.samples.resize(O.nsamp * nbytes);
    MK_CK(cudaMemcpyAsync(O.bwt.data(), dbwt, N, cudaMemcpyDeviceToHost, D.st));
    MK_CK(cudaMemcpyAsync(O.recoded.data(), drec, N, cudaMemcpyDeviceToHost, D.st));
    MK_CK(cudaMemcpyAsync(O.order.data(), dorder, nseq * 4ull, cudaMemcpyDeviceToHost, D.st));
    MK_CK(cudaMemcpyAsync(O.index1.data(), di1, O.index1.size() * 8, cudaMemcpyDeviceToHost, D.st));
    MK_CK(cudaMemcpyAsync(O.index2.data(), di2, O.index2.size() * 2, cudaMemcpyDeviceToHost, D.st));
    if (O.nsamp) MK_CK(cudaMemcpyAsync(O.samples.data(), dsamp, O.samples.size(), cudaMemcpyDeviceToHost, D.st));
    MK_CK(cudaStreamSynchronize(D.st));
    S.assemble_ms = ms_since(t0);
    return KJ_OK;
}

}  // namespace

extern "C" int kj_mkfmi(const char* faa_path, const char* out_prefix, const kj_mkfmi_opts* opts, int device, kj_mkfmi_stats* stats) {
    if (!faa_path || !out_prefix || !*out_prefix) { kj_err() = "kj_mkfmi: null argument"; return KJ_ERR_ARG; }
    const int e = opts ? opts->chpt_exp : 3;
    if (e < 0 || e > 16) { kj_err() = "kj_mkfmi: chpt_exp must be 0..16"; return KJ_ERR_ARG; }
    std::string letters = (opts && opts->alphabet && *opts->alphabet) ? opts->alphabet : "ACDEFGHIKLMNPQRSTVWY";
    if (letters == "protein") letters = "ACDEFGHIKLMNPQRSTVWYX";                                    // mkbwt.c:892
    else if (letters == "DNA" || letters == "RNA") { kj_err() = "kj_mkfmi: nucleotide alphabets are not supported"; return KJ_ERR_UNSUPPORTED; }
    for (size_t i = 0; i < letters.size(); i++) {
        if (!isalpha((unsigned char)letters[i])) { kj_err() = "kj_mkfmi: the alphabet must consist of letters"; return KJ_ERR_ARG; }
        for (size_t j = 0; j < i; j++) if (toupper((unsigned char)letters[j]) == toupper((unsigned char)letters[i])) { kj_err() = "kj_mkfmi: a letter occurs twice in the alphabet"; return KJ_ERR_ARG; }
    }
    if (letters.size() > 24) { kj_err() = "kj_mkfmi: at most 24 letters are supported"; return KJ_ERR_UNSUPPORTED; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) { cudaGetLastError(); kj_err() = "no CUDA device available (this library has no CPU fallback)"; return KJ_ERR_NO_DEVICE; }
    if (device < 0 || device >= ndev) { kj_err() = "kj_mkfmi: no such device"; return KJ_ERR_ARG; }
    kj_mkfmi_stats S; memset(&S, 0, sizeof S);
    auto t0 = clk::now();
    Faa F; int rc = parse_faa(faa_path, letters, F);
    if (rc) return rc;
    S.parse_ms = ms_since(t0);
    S.bwtlen = (int64_t)F.T.size(); S.nseq = (int32_t)F.ids.size();
    if (F.ids.size() >= (1ull << 31)) { kj_err() = "kj_mkfmi: too many sequences"; return KJ_ERR_UNSUPPORTED; }
    const std::string alphabet = "*" + letters;
    Out O;
    {
        if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); kj_err() = "kj_mkfmi: cudaSetDevice failed"; return KJ_ERR_CUDA; }
        Dev D;
        MK_CK(cudaStreamCreateWithFlags(&D.st, cudaStreamNonBlocking));
        rc = build(F, (int)alphabet.size(), e, O, S, D);
        cudaStreamSynchronize(D.st); cudaStreamDestroy(D.st);
        if (rc) return rc;
    }
    t0 = clk::now();
    if ((rc = write_files(out_prefix, F, O, alphabet, e, opts && opts->write_bwt_sa))) return rc;
    S.write_ms = ms_since(t0);
    if (stats) *stats = S;
    return KJ_OK;
}
