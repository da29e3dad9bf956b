// kernels.cuh -- sm_100a kernels of the find-tfbs hot path.
//
//   K0  grouping      sig/group kernels     replaces load_diffs + group_by_diffs      (haplotype.rs:13-75)
//   K1  build         k_ref_prefix, k_walk  replaces patch_haplotype                  (haplotype.rs:94-156): segments + hash
//                     k_emit_list           2-bit packing (+ N mask) of the bases that are scored
//       dedup         k_seq_*               the sequence-keyed map of load_haplotypes (haplotype.rs:81-85)
//   K2  work list     k_items, k_item_*     what has to be scored (find_all_matches, main.rs:94-154; delta scoring, shared items)
//       scan          k_scan                replaces matches / apply_pwm              (pattern.rs:119-171)
//                                           + the hit -> inner-region test            (main.rs:500-505)
//       finish        k_group_finish        inherited / lost reference hits, shared item counts -> per-group count rows
//   BED merge         k_bed_rank/merge      merged regions of all BED files          (bed.rs:37-45, range.rs:43-87)
//   K3  count/rows    k_rows_*              count_matches_by_sample fan-out           (main.rs:506-531)
//                                           + min/max filter of counts_as_genotypes   (main.rs:439-458)
//       attribution   k_att_*               per row, the configurations that change its count (option "attribution")
//       sites         k_site_*              per configuration, the hits it gains and loses (option "sites"), and per record
//                                             alone (option "record_sites")
//
// All arithmetic is integer; results are bit-exact by construction (scores are i32 sums, SURVEY D1).
#pragma once
#include "kernels_base.cuh"
#include "dev_common.cuh"
#include "k0_grouping.cuh"
#include "prefix_scan.cuh"
#include "k1_build.cuh"
#include "k2_types.cuh"
#include "k2_worklist.cuh"
#include "k2c_configs.cuh"
#include "k2_scan.cuh"
#include "k2_finish.cuh"
#include "k3_rows.cuh"
#include "k3_fanout.cuh"
#include "k3_attribution.cuh"
#include "k3_sites.cuh"
#include "k_bed.cuh"
