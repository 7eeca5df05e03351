// Run an ensemble to equilibrium (pmoc_model_equilibrate): chunks of pmoc_model_run over the members still moving,
// each followed by one check kernel that freezes the members whose state has stopped moving and compacts the others
// into the next active list.
//
// Spin-up is what the reference's scripts are mostly run for (run_JansenNadeau_2018.py: 144 000 iterations, then a
// pickup), and members of a sweep settle at very different times.  A frozen member is simply left out of the
// remaining launches: its state, carried streamfunctions and status stay as the chunk that ended at its stop left
// them, which is what pmoc_model_run over the same iterations gives it (split launches and member lists reproduce
// one launch bit for bit).
//
// Compiled as part of the pmoc_ops.cu translation unit (included at its end), not on its own.
#pragma once
#include "pmoc_common.cuh"

namespace pmk {

constexpr int kEqWarps = 8;  // members (one warp each) per CTA of the check
constexpr double kMaxFinite = 1.7976931348623157e308;

// The caller's work buffer, in 8-byte words: the counter, two active lists of M members, then the snapshot of every
// member's state (basin, north, pac columns and the mixed layer's bs, as the model has them).
struct EqLayout {
  long long M, per;  // per: snapshot words per member
  uint64_t bytes() const { return 8ull * (uint64_t)(1 + 2 * M + per * M); }
};

static EqLayout eq_layout(const pmoc_model& m) {
  const unsigned f = m.flags;
  const long long cols = 1 + ((f & PMOC_HAS_NORTH) ? 1 : 0) + ((f & PMOC_HAS_PAC) ? 1 : 0);
  return EqLayout{m.M, cols * m.nz + ((f & PMOC_HAS_ML) ? m.ny : 0)};
}

struct EqArgs {
  pmoc_model m;
  MemberList list;  // the members of the chunk just run (NULL: every member)
  double tol;
  long long it;     // the iteration the chunk ended at
  int first;        // take the first snapshot only
  long long per;
  double* snap;
  int64_t* next;    // the next active list ...
  unsigned long long* count;  // ... and its length
  int64_t* stopped_at;
  uint8_t* converged;
};

// One warp per member of the list: |b_now - b_prev| <= tol everywhere (IEEE subtraction, fabs and comparison only,
// so numpy reproduces the decision), any non-finite value stops the member as not converged; the snapshot is
// refreshed and the members still moving are appended to the next list (in no particular order).
PM_GLOBAL void k_equil_check(EqArgs a) {
  const pmoc_model& M = a.m;
  const long long slot = rt::block_idx() * rt::warps_per_block() + rt::warp_in_block();
  if (slot >= a.list.slots(M.M)) return;
  const long long m = a.list.members ? a.list.members[slot] : slot;
  const int L = rt::lane(), nz = M.nz;
  double* snap = a.snap + m * a.per;
  bool moved = false, bad = false;
  auto visit = [&](const double* now, int n, int off) {
    for (int i = L; i < n; i += 32) {
      const double v = now[i];
      moved |= !(fabs(v - snap[off + i]) <= a.tol);
      bad |= !(fabs(v) <= kMaxFinite);
      snap[off + i] = v;
    }
  };
  int off = 0;
  visit(M.basin.b + m * nz, nz, off);
  off += nz;
  if (M.flags & PMOC_HAS_NORTH) {
    visit(M.north.b + m * nz, nz, off);
    off += nz;
  }
  if (M.flags & PMOC_HAS_PAC) {
    visit(M.pac.b + m * nz, nz, off);
    off += nz;
  }
  if (M.flags & PMOC_HAS_ML) visit(M.ml_bs + m * M.ny, M.ny, off);
  const bool mv = rt::ballot(moved) != 0, nf = rt::ballot(bad) != 0;
  if (L != 0) return;
  a.stopped_at[m] = a.it;
  if (a.first) {
    a.converged[m] = 0;
  } else if (nf || !mv) {
    a.converged[m] = nf ? 0 : 1;
  } else {
    a.next[rt::atomic_add_global(a.count, 1ull)] = m;
  }
}

int check_equilibrate(const pmoc_model* m, int64_t it0, int64_t max_steps, int64_t every, double tol,
                      const void* stopped_at, const void* converged) {
  if (int rc = check_model(m)) return rc;
  if (it0 < 0 || max_steps < 0) return fail(PMOC_EINVAL, "negative it0 / max_steps");
  if (every <= 0 || every % m->K != 0) return fail(PMOC_EINVAL, "every must be a positive multiple of K");
  if (max_steps % m->K != 0) return fail(PMOC_EINVAL, "max_steps must be a multiple of K");
  if (!(tol >= 0.0)) return fail(PMOC_EINVAL, "tol must be >= 0");
  if (!stopped_at || !converged) return fail(PMOC_EINVAL, "stopped_at / converged is NULL");
  return PMOC_OK;
}

}  // namespace pmk

extern "C" {

uint64_t pmoc_equilibrate_work_bytes(const pmoc_model* m) {
  if (!m || m->M <= 0 || m->nz < 0 || m->ny < 0) return 0;
  return eq_layout(*m).bytes();
}

int pmoc_model_equilibrate(const pmoc_model* m, int64_t it0, int64_t max_steps, int64_t every, double tol,
                           int64_t* stopped_at, uint8_t* converged, void* work, uint64_t work_bytes, void* stream) {
  if (int rc = check_equilibrate(m, it0, max_steps, every, tol, stopped_at, converged)) return rc;
  const EqLayout lay = eq_layout(*m);
  if (!work || work_bytes < lay.bytes()) return fail(PMOC_EINVAL, "work needs pmoc_equilibrate_work_bytes() bytes");
  EqArgs a;
  a.m = *m;
  a.list = MemberList{nullptr, 0};
  a.tol = tol;
  a.it = it0;
  a.first = 1;
  a.per = lay.per;
  a.count = static_cast<unsigned long long*>(work);
  int64_t* lists = reinterpret_cast<int64_t*>(a.count + 1);
  a.snap = reinterpret_cast<double*>(lists + 2 * lay.M);
  a.stopped_at = stopped_at;
  a.converged = converged;
  a.next = lists;
  const int block = 32 * kEqWarps;
  if (int rc = launch(k_equil_check, (lay.M + kEqWarps - 1) / kEqWarps, block, 0, stream, a)) return rc;
  a.first = 0;
  // Every member is active until the first check; a list that holds every member runs as pmoc_model_run (the same
  // bits, the launch of a plain run).
  const int64_t* list = nullptr;
  unsigned long long n = (unsigned long long)lay.M;
  int which = 0;
  for (long long it = it0, end = it0 + max_steps; it < end && n > 0;) {
    const long long len = every < end - it ? every : end - it;
    const int rc = list ? pmoc_model_run_members(m, list, (int64_t)n, it, len, stream)
                        : pmoc_model_run(m, it, len, stream);
    if (rc) return rc;
    it += len;
    a.list = MemberList{list, (long long)n};
    a.it = it;
    a.next = lists + which * lay.M;
    PM_CUDA_OK(cudaMemsetAsync(a.count, 0, sizeof(unsigned long long), (cudaStream_t)stream));
    if (int rc2 = launch(k_equil_check, ((long long)n + kEqWarps - 1) / kEqWarps, block, 0, stream, a)) return rc2;
    PM_CUDA_OK(cudaMemcpyAsync(&n, a.count, sizeof(n), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    PM_CUDA_OK(cudaStreamSynchronize((cudaStream_t)stream));
    list = n == (unsigned long long)lay.M ? nullptr : a.next;
    which ^= 1;
  }
  return PMOC_OK;
}

}  // extern "C"
