// Host-built "plan" that maps the reference's four wave types (Rc, Rg, Lc, Lg;
// /root/reference/src/SWD/surfdisp.cpp:190-297) onto unique period sequences and eigen solves.
// Shared by the two translation units (capi.cu, swd_roots_tu.cu).
#pragma once
#include "swd_roots.cuh"

namespace rfs {

#define RFS_MAX_SEQ 12
#define RFS_MAX_ROWS 4

// one requested data block ("row"): a wave type on a period list
struct SwdRow {
  int type;      // 0 Rc, 1 Rg, 2 Lc, 3 Lg
  int nper;      // periods
  int per_off;   // offset of its period list in the period table
  int s0, s1, s2;  // sequences: T, 1.05 T, 0.95 T (s1,s2 = -1 for phase velocity)
  int d_off;     // offset of this row in the concatenated data vector
};

struct SwdPlan {
  int nseq, nrow;
  int nsolve;  // total (sequence, period) pairs == total periods over sequences
  int ndata;   // total data count over rows
  int nmode;   // modes solved (mode+1); the last one is reported
  SwdSeq seq[RFS_MAX_SEQ];
  SwdRow row[RFS_MAX_ROWS];
};

// Per-set period lists (rfs_config_obs_periods): observation set s observes a subset of the plan's
// period grid, and every (model, sequence) job of a row of set s runs set s's compact list.  Results
// keep the plan's capacity layout: compact period k of sequence q is solve plan.seq[q].out_off + k.
// tab [nsets][ld] ints, ld = 2 nseq + 2 ndata, per set:
//   [0, nseq)              per_off of sequence q's compact list in the period table
//   [nseq, 2 nseq)         its length (0: the set observes none of the sequence's periods)
//   [2 nseq + d_off + k]   row r's compact period k -> grid position (d_off = plan.row[r].d_off)
//   [2 nseq + ndata + j]   grid position j of the data vector observed (1) or not (0)
// tab == NULL, or a row whose set index lies outside [0, nsets): the plan's own lists (such a row is
// failed by the residual kernels).  One code path for both is what makes an all-ones table give the
// bits of no table.
struct SwdSetView {
  const int *tab;
  const int *set;  // [B] set index of each row of the launch, or NULL (set 0)
  int nsets, ld;
  RFS_DEVINL const int *of(long long b) const {
    if (!tab) return nullptr;
    const int s = set ? set[b] : 0;
    return (s >= 0 && s < nsets) ? tab + (long long)s * ld : nullptr;
  }
  // sequence q of row b's job
  RFS_DEVINL SwdSeq seq(const SwdPlan &P, int q, long long b) const {
    SwdSeq sq = P.seq[q];
    if (const int *t = of(b)) {
      sq.per_off = t[q];
      sq.nper = t[P.nseq + q];
    }
    return sq;
  }
  // data row r of row b: its compact length and period offset; *c2g = compact -> grid map (NULL: identity)
  RFS_DEVINL SwdRow row(const SwdPlan &P, int r, long long b, const int **c2g) const {
    SwdRow rw = P.row[r];
    *c2g = nullptr;
    if (const int *t = of(b)) {
      rw.per_off = t[rw.s0];
      rw.nper = t[P.nseq + rw.s0];
      *c2g = t + 2 * P.nseq + rw.d_off;
    }
    return rw;
  }
};

}  // namespace rfs
