// Launchers of the TAD engine kernels (implemented in tad_kernels.cu, tad_spill.cu, tad_arima.cu).
#pragma once
#include "tad_common.cuh"

namespace tad {

cudaError_t launch_hist(cudaStream_t st, const ColPtrs &c, uint64_t R, const RowFilter &f, int logB, uint32_t *hist);
// slot_cap == 0: exact mode, cursor[] holds absolute row cursors (from the bucket scan).
// slot_cap  > 0: optimistic mode, cursor[] counts arrivals from zero, bucket b owns part[b * slot_cap ...); rows past the
//                slot go to ovf[] (ovf_count may exceed ovf_cap: the caller then falls back to the exact partition).
cudaError_t launch_scatter(cudaStream_t st, const ColPtrs &c, uint64_t R, const RowFilter &f, int logB, uint32_t *cursor,
                           Row32 *part, uint32_t slot_cap = 0, Row32 *ovf = nullptr, uint32_t ovf_cap = 0,
                           uint32_t *ovf_count = nullptr);
cudaError_t launch_bucket_scan(cudaStream_t st, const uint32_t *hist, uint32_t *offsets, uint32_t *cursor, uint32_t B,
                               uint32_t cap, uint32_t *big_list, uint32_t *big_base, uint32_t *cls_list /* 3 x B or null */,
                               uint32_t *stats, void *scan_sync, uint32_t epoch);
size_t scan_sync_bytes();   // zero-initialised once; epoch must be > 0 and differ between launches
// csr_p != nullptr: also rank every series by value and write the permutation (value rank -> time
// index) the DBSCAN detector sweeps over.
// `offsets` are the (virtual, contiguous) bucket offsets used for entries / csr arrays; the rows
// themselves are read through `seg`.
cudaError_t launch_group(cudaStream_t st, const SegDesc &seg, SeriesEntry *entries, const uint32_t *offsets, uint32_t B,
                         const uint32_t *cls_list, const uint32_t n_cls[3], uint64_t *csr_v, uint32_t *csr_t,
                         uint32_t *csr_p, uint32_t *nsb, uint32_t *npb, int reducer, int *launches);
cudaError_t launch_series_scan(cudaStream_t st, const uint32_t *nsb, const uint32_t *npb, uint32_t *sbase, uint32_t B,
                               uint32_t *stats, void *scan_sync, uint32_t epoch);
cudaError_t launch_detect_ewma(cudaStream_t st, const SeriesEntry *entries, const uint32_t *offsets, const uint32_t *sbase, uint32_t B,
                               uint32_t S, const uint64_t *csr_v, const uint32_t *csr_t, const OutCols &out,
                               uint32_t out_cap, uint32_t *stats, int emit_all);
cudaError_t launch_detect_dbscan(cudaStream_t st, const SeriesEntry *entries, const uint32_t *offsets, const uint32_t *sbase,
                                 uint32_t B, uint32_t S, const uint64_t *csr_v, const uint32_t *csr_t, const uint32_t *csr_p,
                                 uint32_t *scratch_pc, uint8_t *scratch_flag, const OutCols &out, uint32_t out_cap,
                                 uint32_t *stats, int emit_all);

// ARIMA (tad_arima.cu): Box-Cox + per-prefix ARIMA(1,1,1) MLE fits (when `fit`) then score/flag/compact.
// scratch_y / scratch_pred: one double per point slot; scratch_lam: one double per series.
cudaError_t launch_detect_arima(cudaStream_t st, const SeriesEntry *entries, const uint32_t *offsets, const uint32_t *sbase,
                                uint32_t B, uint32_t S, const uint64_t *csr_v, const uint32_t *csr_t, double *scratch_y,
                                double *scratch_pred, double *scratch_lam, bool fit, const OutCols &out, uint32_t out_cap,
                                uint32_t *stats, int emit_all);

// Oversized buckets (more rows than the shared-memory capacity): global-memory path.
// Sorts the rows of all listed buckets by (hash, key, time), reduces duplicates and writes the
// same per-series arrays / in-place series entries / nsb / npb the group kernel produces.
// `scratch` must hold spill_scratch_bytes(big_rows) bytes.  Returns launches through *launches.
size_t spill_scratch_bytes(uint64_t big_rows);
// Sort a capacity-class bucket list ascending (CUB radix sort over `key_bits` bits); scratch from sort_lists_scratch_bytes(max n).
size_t sort_lists_scratch_bytes(uint32_t max_items);
cudaError_t sort_bucket_list(cudaStream_t st, uint32_t *list, uint32_t n, int key_bits, void *scratch, size_t scratch_bytes);
// Optimistic partition (seg.stride != 0): a listed bucket holds min(count, stride) rows in its slot and the rest in
// ovf[0, n_ovf) (every overflow row belongs to a listed bucket).
cudaError_t run_spill(cudaStream_t st, const SegDesc &seg, SeriesEntry *entries, const uint32_t *offsets, const uint32_t *big_list,
                      const uint32_t *big_base, uint32_t n_big, uint64_t big_rows, void *scratch, size_t scratch_bytes,
                      uint64_t *csr_v, uint32_t *csr_t, uint32_t *nsb, uint32_t *npb, int reducer, int *launches,
                      const Row32 *ovf = nullptr, uint32_t n_ovf = 0);

}  // namespace tad

namespace tad {
// Multi-GPU, optimistic partition: pc.p[s] = source rank s's arrival counters (its own for s = me, IPC-mapped otherwise).
// Fills cnt[world x B_local] / total[B_local] for the owned bucket range and adds the sum of this rank's own B_global
// counters (= its rows that passed the filters) to *kept_out.  Two launches.
struct PeerCounters { const uint32_t *p[8]; };
cudaError_t launch_gather_counts(cudaStream_t st, const PeerCounters &pc, int world, uint32_t b_lo, uint32_t B_local, uint32_t slot,
                                 uint32_t *cnt, uint32_t *total, const uint32_t *my_counters, uint32_t B_global, uint32_t *kept_out);
// Multi-GPU: per-source segment offsets and total bucket sizes of this rank's bucket range from the
// all-gathered histograms.  hist_all[r * B_global + b]; range = [b_lo, b_lo + B_local).
cudaError_t launch_segment_scan(cudaStream_t st, const uint32_t *hist_all, uint32_t B_global, uint32_t b_lo, uint32_t B_local,
                                int nseg, uint32_t *seg_off /* nseg x (B_local+1) */, uint32_t *total /* B_local */,
                                unsigned long long *seg_rows /* nseg */,
                                unsigned long long *seg_before = nullptr /* nseg: rows of each source in front of the owned range */);
}
