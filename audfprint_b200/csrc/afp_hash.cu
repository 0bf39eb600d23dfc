// K3 — peak-pair fan-out, 20-bit hash packing, cross-shift merge/sort/dedupe.
//
// Replaces Analyzer.peaks2landmarks (audfprint_analyze.py:310-343),
// landmarks2hashes (:81-96) and the concatenate / sort / unique tail of
// wavfile2hashes (:401-422).
//
// Layout trick: every (item, column) owns maxpks fixed peak slots (bins
// ascending) and every peak owns `fanout` hash slots, so no prefix sums are
// needed until the very end.  All hashes of one file that carry the same time
// value live in the same column of its (up to `shifts`) items; the final
// (time, hash)-sorted, de-duplicated output of a file is therefore the
// concatenation over columns of the sorted unique union of at most
// shifts*maxpks*fanout slot values — a per-thread insertion sort.
#include "afp_internal.cuh"

namespace {

struct HashArgs {
  const ItemDesc* items;
  int item0;
  int nitems, nfiles, shifts, maxpks, fanout, targetdf, mindt, targetdt;
  const uint8_t* pk_bin;
  const uint8_t* pk_cnt;
  const int32_t* item_scols;
  uint32_t* lm;                 // [frames][maxpks][fanout]
  const int64_t* file_col_base; // [nfiles+1]
  int64_t total_cols;
  int32_t* col_cnt;             // [total_cols] counts, then exclusive per-file offsets
  int32_t* file_tot;            // [nfiles]
  const int64_t* file_off;      // [nfiles+1]
  int32_t* hashes;              // [total][2]
};

// One CTA per item.  The item's peaks are first compacted (window by window) into a
// shared-memory list sorted by (column, bin) — the order the reference visits them in —
// then one thread per SOURCE PEAK scans the following list entries: ~18 candidates on
// average instead of 61 mostly-empty columns, and no thread is spent on empty slots.
// The hash slots of `lm` are pre-filled with AFP_NO_HASH by a memset.
constexpr int LM_THREADS = 256;
constexpr int PCAP = 11264;   // peak entries per window ((col - w0):20 | slot:4 | bin:8)

__global__ void __launch_bounds__(LM_THREADS) afp_landmark_kernel(HashArgs a) {
  __shared__ uint32_t s_pk[PCAP];
  __shared__ int s_scan[LM_THREADS];
  __shared__ int s_run;
  const ItemDesc it = a.items[a.item0 + blockIdx.x];
  const int scols = a.item_scols[a.item0 + blockIdx.x];   // last peak column + 1 (:321)
  const int P = a.maxpks, F = a.fanout, tid = threadIdx.x;
  const int64_t base = it.frame_base;
  // Columns are stored relative to the window start: a window spans at most W + targetdt < 2^20 columns,
  // while an item may have any int32 number of frames.
  const int W = max(64, PCAP / P - a.targetdt - 1);       // source columns per window
  for (int w0 = 0; w0 < scols; w0 += W) {
    const int wend = min(scols, w0 + W + a.targetdt);     // sources in [w0, w0+W), targets up to +targetdt
    if (tid == 0) s_run = 0;
    __syncthreads();
    for (int c0 = w0; c0 < wend; c0 += LM_THREADS) {      // compaction, column order
      const int c = c0 + tid;
      const int n = (c < wend) ? a.pk_cnt[base + c] : 0;
      s_scan[tid] = n;
      __syncthreads();
      for (int o = 1; o < LM_THREADS; o <<= 1) {
        const int v = (tid >= o) ? s_scan[tid - o] : 0;
        __syncthreads();
        s_scan[tid] += v;
        __syncthreads();
      }
      const int at = s_run + s_scan[tid] - n;
      for (int k = 0; k < n; ++k)
        s_pk[at + k] = ((uint32_t)(c - w0) << 12) | ((uint32_t)k << 8) | a.pk_bin[(base + c) * P + k];
      __syncthreads();
      if (tid == LM_THREADS - 1) s_run += s_scan[tid];
      __syncthreads();
    }
    const int np = s_run;
    for (int i = tid; i < np; i += LM_THREADS) {
      const uint32_t e = s_pk[i];
      const int col = w0 + (int)(e >> 12), slot = (int)((e >> 8) & 15), b1 = (int)(e & 255);
      if (col >= w0 + W) break;                           // entries are column-sorted: only targets remain
      uint32_t* out = a.lm + ((base + col) * P + slot) * F;
      const int c2lo = col + a.mindt, c2hi = min(scols, col + a.targetdt);     // :331-332
      int n = 0;
      for (int j = (a.mindt > 0) ? i + 1 : i - slot; j < np && n < F; ++j) {
        const uint32_t t = s_pk[j];
        const int c2 = w0 + (int)(t >> 12);
        if (c2 >= c2hi) break;
        if (c2 < c2lo) continue;
        const int b2 = (int)(t & 255);
        if (abs(b2 - b1) < a.targetdf)                                          // :335
          out[n++] = ((uint32_t)(b1 & 0xFF) << 12) | ((uint32_t)((b2 - b1) & 0x3F) << 6) |
                     (uint32_t)((c2 - col) & 0x3F);                             // :92-95
      }
    }
    __syncthreads();
  }
}

__device__ __forceinline__ int find_file(const int64_t* fcb, int nfiles, int64_t gcol) {
  int lo = 0, hi = nfiles;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (fcb[mid] <= gcol) lo = mid; else hi = mid;
  }
  return lo;
}

// Sorted unique union of the hash slots of one (file, column) over all shifts.
template <bool WRITE>
__global__ void __launch_bounds__(128) afp_merge_kernel(HashArgs a) {
  const int64_t gcol = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gcol >= a.total_cols) return;
  const int f = find_file(a.file_col_base, a.nfiles, gcol);
  const int col = (int)(gcol - a.file_col_base[f]);
  uint32_t buf[AFP_MAX_MERGE];
  int n = 0;
  const int PF = a.maxpks * a.fanout;
  for (int s = 0; s < a.shifts; ++s) {
    const ItemDesc it = a.items[f * a.shifts + s];
    if (col >= it.nframes) continue;
    if (a.pk_cnt[it.frame_base + col] == 0) continue;
    const uint32_t* src = a.lm + (it.frame_base + col) * PF;
    for (int e = 0; e < PF; ++e) {
      const uint32_t h = src[e];
      if (h == AFP_NO_HASH) continue;
      int i = n;
      while (i > 0 && buf[i - 1] > h) --i;
      if (i > 0 && buf[i - 1] == h) continue;        // duplicate across shifts (:417)
      for (int k = n; k > i; --k) buf[k] = buf[k - 1];
      buf[i] = h;
      ++n;
    }
  }
  if (!WRITE) {
    a.col_cnt[gcol] = n;
  } else {
    int32_t* out = a.hashes + 2 * (a.file_off[f] + a.col_cnt[gcol]);
    for (int i = 0; i < n; ++i) {
      out[2 * i] = col;
      out[2 * i + 1] = (int32_t)buf[i];
    }
  }
}

// In-place exclusive scan of col_cnt inside each file; file totals out.
__global__ void __launch_bounds__(256) afp_file_scan_kernel(HashArgs a) {
  __shared__ int s_scan[256];
  __shared__ int s_run;
  const int f = blockIdx.x, tid = threadIdx.x;
  const int64_t c0 = a.file_col_base[f];
  const int ncol = (int)(a.file_col_base[f + 1] - c0);
  if (tid == 0) s_run = 0;
  __syncthreads();
  for (int t0 = 0; t0 < ncol; t0 += 256) {
    const int t = t0 + tid;
    const int c = (t < ncol) ? a.col_cnt[c0 + t] : 0;
    s_scan[tid] = c;
    __syncthreads();
    for (int o = 1; o < 256; o <<= 1) {
      const int v = (tid >= o) ? s_scan[tid - o] : 0;
      __syncthreads();
      s_scan[tid] += v;
      __syncthreads();
    }
    if (t < ncol) a.col_cnt[c0 + t] = s_scan[tid] - c + s_run;
    __syncthreads();
    if (tid == 255) s_run += s_scan[255];
    __syncthreads();
  }
  if (tid == 0) a.file_tot[f] = s_run;
}

// Single-CTA exclusive scan int32[n] -> int64[n+1].
__global__ void __launch_bounds__(1024) afp_scan_kernel(const int32_t* in, int64_t* out, int64_t n) {
  __shared__ long long s_scan[1024];
  __shared__ long long s_run;
  const int tid = threadIdx.x;
  if (tid == 0) s_run = 0;
  __syncthreads();
  for (int64_t i0 = 0; i0 < n; i0 += 1024) {
    const int64_t i = i0 + tid;
    const long long c = (i < n) ? in[i] : 0;
    s_scan[tid] = c;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
      const long long v = (tid >= o) ? s_scan[tid - o] : 0;
      __syncthreads();
      s_scan[tid] += v;
      __syncthreads();
    }
    if (i < n) out[i] = s_scan[tid] - c + s_run;
    __syncthreads();
    if (tid == 1023) s_run += s_scan[1023];
    __syncthreads();
  }
  if (tid == 0) out[n] = s_run;
}

// ---- explicit peak list -> landmark rows (Analyzer.peaks2landmarks as a call) ---
__global__ void afp_scatter_peaks_kernel(const int32_t* rows, int64_t n, int maxpks, int T, uint8_t* pk_bin,
                                         uint8_t* pk_cnt, int* err) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int col = rows[2 * i], bin = rows[2 * i + 1];
  if (col < 0 || col >= T || bin < 0 || bin >= AFP_NBINS) { atomicExch(err, 1); return; }
  if (i > 0 && (rows[2 * (i - 1)] > col || (rows[2 * (i - 1)] == col && rows[2 * (i - 1) + 1] >= bin))) {
    atomicExch(err, 2);   // not sorted column-major / bins ascending
    return;
  }
  int slot = 0;
  while (i - slot - 1 >= 0 && rows[2 * (i - slot - 1)] == col) {
    ++slot;
    if (slot >= maxpks) { atomicExch(err, 3); return; }
  }
  pk_bin[(int64_t)col * maxpks + slot] = (uint8_t)bin;
  if (i == n - 1 || rows[2 * (i + 1)] != col) pk_cnt[col] = (uint8_t)(slot + 1);
}

template <bool WRITE>
__global__ void afp_lm_rows_kernel(const uint32_t* lm, int T, int PF, int32_t* col_cnt, int32_t* out) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= T) return;
  const uint32_t* src = lm + (int64_t)col * PF;
  int n = 0;
  int32_t* dst = WRITE ? out + 4 * (int64_t)col_cnt[col] : nullptr;
  for (int e = 0; e < PF; ++e) {
    const uint32_t h = src[e];
    if (h == AFP_NO_HASH) continue;
    if (WRITE) {   // inverse packing, audfprint_analyze.py:99-112
      const int b1 = (h >> 12) & 0xFF;
      int df = (h >> 6) & 0x3F;
      if (df >= 32) df -= 64;
      dst[4 * n] = col; dst[4 * n + 1] = b1; dst[4 * n + 2] = b1 + df; dst[4 * n + 3] = h & 0x3F;
    }
    ++n;
  }
  if (!WRITE) col_cnt[col] = n;
}

}  // namespace

// Runs landmark -> count -> scans.  The write pass needs the total (to size the
// output) and is issued by afp_finish_hashes.
static HashArgs make_args(afp_ctx* c) {
  HashArgs a;
  a.items = c->d_items.as<ItemDesc>();
  a.item0 = 0;
  a.nitems = c->nitems;
  a.nfiles = c->nfiles;
  a.shifts = c->ap.shifts;
  a.maxpks = c->ap.maxpksperframe;
  a.fanout = c->ap.maxpairsperpeak;
  a.targetdf = c->ap.targetdf;
  a.mindt = c->ap.mindt;
  a.targetdt = c->ap.targetdt;
  a.pk_bin = c->d_pk_bin.as<uint8_t>();
  a.pk_cnt = c->d_pk_cnt.as<uint8_t>();
  a.item_scols = c->d_item_scols.as<int32_t>();
  a.lm = c->d_lm.as<uint32_t>();
  a.file_col_base = c->d_file_col_base.as<int64_t>();
  a.total_cols = c->total_cols;
  a.col_cnt = c->d_col_cnt.as<int32_t>();
  a.file_tot = c->d_file_tot.as<int32_t>();
  a.file_off = c->d_file_off.as<int64_t>();
  a.hashes = c->d_hashes.as<int32_t>();
  return a;
}

int afp_landmarks_from_peaks_impl(afp_ctx* c, const int32_t* rows_in, int64_t n, int on_host, int64_t* nlm) {
  c->batch_valid = false;
  c->nlandmarks = -1;
  if (n == 0) { c->nlandmarks = 0; if (nlm) *nlm = 0; return AFP_OK; }
  const int32_t* drows = rows_in;
  int32_t last[2];
  if (on_host) {
    AFP_CUDA(c, c->d_q.reserve(sizeof(int32_t) * 2 * (size_t)n));
    AFP_CUDA(c, cudaMemcpyAsync(c->d_q.p, rows_in, sizeof(int32_t) * 2 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    drows = c->d_q.as<int32_t>();
    last[0] = rows_in[2 * (n - 1)];
  } else {
    AFP_CUDA(c, cudaMemcpyAsync(last, rows_in + 2 * (n - 1), sizeof(last), cudaMemcpyDeviceToHost, c->stream));
    AFP_CUDA(c, cudaStreamSynchronize(c->stream));
  }
  if (last[0] < 0 || last[0] > (1 << 28)) AFP_FAIL(c, AFP_ERR_INVALID, "bad peak column");
  const int T = last[0] + 1;   // scols = last peak column + 1 (:321)
  const size_t P = (size_t)c->ap.maxpksperframe, F = (size_t)c->ap.maxpairsperpeak, fr = (size_t)T + 1;
  ItemDesc it{};
  it.nframes = T;
  AFP_CUDA(c, c->d_items.reserve(sizeof(ItemDesc) * 2));
  AFP_CUDA(c, c->d_pk_bin.reserve(P * fr));
  AFP_CUDA(c, c->d_pk_cnt.reserve(fr));
  AFP_CUDA(c, c->d_item_scols.reserve(sizeof(int32_t) * 2));
  AFP_CUDA(c, c->d_lm.reserve(sizeof(uint32_t) * P * F * fr));
  AFP_CUDA(c, c->d_col_cnt.reserve(sizeof(int32_t) * fr));
  AFP_CUDA(c, c->d_file_tot.reserve(sizeof(int32_t) * 4));
  AFP_CUDA(c, c->d_file_col_base.reserve(sizeof(int64_t) * 2));
  AFP_CUDA(c, c->d_tmp.reserve(64));
  const int64_t fcb[2] = {0, T};
  AFP_CUDA(c, cudaMemcpyAsync(c->d_items.p, &it, sizeof(it), cudaMemcpyHostToDevice, c->stream));
  AFP_CUDA(c, cudaMemcpyAsync(c->d_file_col_base.p, fcb, sizeof(fcb), cudaMemcpyHostToDevice, c->stream));
  AFP_CUDA(c, cudaMemcpyAsync(c->d_item_scols.p, &T, sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
  AFP_CUDA(c, cudaMemsetAsync(c->d_pk_cnt.p, 0, fr, c->stream));
  AFP_CUDA(c, cudaMemsetAsync(c->d_tmp.p, 0, sizeof(int), c->stream));
  afp_scatter_peaks_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(
      drows, n, (int)P, T, c->d_pk_bin.as<uint8_t>(), c->d_pk_cnt.as<uint8_t>(), c->d_tmp.as<int>());
  AFP_CUDA(c, cudaGetLastError());
  c->launches++;
  c->nfiles = 1; c->nitems = 1; c->total_frames = T; c->total_cols = T;
  HashArgs a = make_args(c);
  AFP_CUDA(c, cudaMemsetAsync(c->d_lm.p, 0xFF, sizeof(uint32_t) * P * F * fr, c->stream));
  afp_landmark_kernel<<<1, LM_THREADS, 0, c->stream>>>(a);
  AFP_CUDA(c, cudaGetLastError());
  afp_lm_rows_kernel<false><<<(T + 127) / 128, 128, 0, c->stream>>>(a.lm, T, (int)(P * F), a.col_cnt, nullptr);
  AFP_CUDA(c, cudaGetLastError());
  afp_file_scan_kernel<<<1, 256, 0, c->stream>>>(a);
  AFP_CUDA(c, cudaGetLastError());
  c->launches += 3;
  int32_t total = 0;
  int err = 0;
  AFP_CUDA(c, cudaMemcpyAsync(&total, c->d_file_tot.p, sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
  AFP_CUDA(c, cudaMemcpyAsync(&err, c->d_tmp.p, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  AFP_CUDA(c, cudaStreamSynchronize(c->stream));
  if (err == 3) AFP_FAIL(c, AFP_ERR_UNSUPPORTED, "more peaks in one column than maxpksperframe");
  if (err) AFP_FAIL(c, AFP_ERR_INVALID, "peak rows must be (col, bin) in [0,T)x[0,256), column-major, bins ascending");
  AFP_CUDA(c, c->d_hashes.reserve(sizeof(int32_t) * 4 * (size_t)(total + 1)));
  if (total > 0) {
    afp_lm_rows_kernel<true><<<(T + 127) / 128, 128, 0, c->stream>>>(a.lm, T, (int)(P * F), a.col_cnt,
                                                                    c->d_hashes.as<int32_t>());
    AFP_CUDA(c, cudaGetLastError());
    c->launches++;
  }
  c->nlandmarks = total;
  if (nlm) *nlm = total;
  return AFP_OK;
}

int afp_launch_scan_i32_to_i64(afp_ctx* c, const int32_t* in, int64_t* out, int64_t n) {
  afp_scan_kernel<<<1, 1024, 0, c->stream>>>(in, out, n);
  AFP_CUDA(c, cudaGetLastError());
  c->launches++;
  return AFP_OK;
}

int afp_launch_landmarks(afp_ctx* c, int item0, int nitems) {
  if (nitems <= 0 || c->total_frames == 0) return AFP_OK;
  HashArgs a = make_args(c);
  a.item0 = item0;
  {   // empty hash slots = AFP_NO_HASH (0xFFFFFFFF): byte fill of this launch's slot range
    const ItemDesc& i0 = c->h_items[item0];
    const ItemDesc& i1 = c->h_items[item0 + nitems - 1];
    const size_t per_frame = (size_t)c->ap.maxpksperframe * c->ap.maxpairsperpeak * sizeof(uint32_t);
    const size_t f0 = (size_t)i0.frame_base, f1 = (size_t)i1.frame_base + i1.nframes;
    if (f1 > f0) AFP_CUDA(c, cudaMemsetAsync((char*)c->d_lm.p + f0 * per_frame, 0xFF, (f1 - f0) * per_frame, c->stream));
  }
  afp_landmark_kernel<<<nitems, LM_THREADS, 0, c->stream>>>(a);
  AFP_CUDA(c, cudaGetLastError());
  c->launches++;
  return AFP_OK;
}

int afp_launch_hashes(afp_ctx* c) {
  if (c->nfiles == 0) return AFP_OK;
  HashArgs a = make_args(c);
  if (c->total_cols > 0) {
    afp_merge_kernel<false><<<(unsigned)((c->total_cols + 127) / 128), 128, 0, c->stream>>>(a);
    AFP_CUDA(c, cudaGetLastError());
    c->launches++;
  }
  afp_file_scan_kernel<<<c->nfiles, 256, 0, c->stream>>>(a);
  AFP_CUDA(c, cudaGetLastError());
  c->launches++;
  return afp_launch_scan_i32_to_i64(c, c->d_file_tot.as<int32_t>(), c->d_file_off.as<int64_t>(), c->nfiles);
}

int afp_write_hashes(afp_ctx* c) {
  if (c->total_cols == 0) return AFP_OK;
  HashArgs a = make_args(c);
  afp_merge_kernel<true><<<(unsigned)((c->total_cols + 127) / 128), 128, 0, c->stream>>>(a);
  AFP_CUDA(c, cudaGetLastError());
  c->launches++;
  return AFP_OK;
}
