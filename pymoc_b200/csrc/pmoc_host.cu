// Host-buffer entry points and the FP64 roofline probe.
//
// The stateless call (pmoc_model_run_host) and the persistent handle (pmoc_host_open / step / close) share one
// device mirror of the caller's host arrays.  Every per-member array of the mirror carries a class bitmask; a
// call names the classes that go up before its launches and come back after them, and one block loop moves
// them (Mirror::pass, with Mirror::copy).  The emulator build runs this same code on host stand-ins of the
// CUDA runtime calls (pmoc_rt.cuh).
#include "pmoc_common.cuh"

#include <algorithm>
#include <mutex>
#include <new>
#include <vector>

static thread_local unsigned long long g_h2d_bytes = 0, g_d2h_bytes = 0;

extern "C" void pmoc_host_last_bytes(uint64_t* h2d, uint64_t* d2h) {
  if (h2d) *h2d = g_h2d_bytes;
  if (d2h) *d2h = g_d2h_bytes;
}

namespace {

// Mirrors the host arrays of a pmoc_model on the device, and pipelines a call over blocks of members: block c's
// host->device copies, kernel and device->host copies are queued on stream c % kStreams, so the copies of one
// block overlap the kernel of another (members are independent).
constexpr int kStreams = 3;
#ifndef PMOC_HOST_BLOCK_MEMBERS
#define PMOC_HOST_BLOCK_MEMBERS 4096  // 16 blocks for the 65,536-member bench: fill/drain of the pipeline ~6 % of the copies
#endif

// Classes besides the public PMOC_IO_STATE / PSI / DIAG, which pmoc_host_step rejects: the per-member parameter
// vectors, and the arrays every stepping launch writes whether or not it diagnoses (ml_Psi_s, also DIAG).
constexpr unsigned kIoParam = 8u, kIoStepped = 16u;

struct Mirror {
  struct Field {
    char* host;        // host base
    char* dev;         // device base
    size_t slot;       // byte offset of the pointer inside pmoc_model
    size_t per_member; // bytes per member; 0 = shared by all members
    size_t bytes;      // total bytes
    unsigned cat;      // class bits of a per-member array
  };
  cudaStream_t s[kStreams] = {};
  cudaEvent_t shared_ready = nullptr;
  std::vector<Field> fields;
  std::vector<void*> allocs;
  cudaError_t err = cudaSuccess;
  pmoc_model d;       // the caller's model with the device pointers
  cudaMemPool_t pool = nullptr;
  bool fresh = true;  // nothing uploaded yet

  // Streams, event and the library's own memory pool.  The pool is private (one per device, created on first
  // use, kept for the life of the process with its memory retained between calls): the embedding application's
  // default pool is not touched.
  cudaError_t init() {
    static cudaMemPool_t pools[64] = {};
    static std::mutex pools_lock;  // (callers on different threads may open their first handle at the same time)
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
    std::lock_guard<std::mutex> guard(pools_lock);
    if (!pools[dev]) {
      cudaMemPoolProps props = {};
      props.allocType = cudaMemAllocationTypePinned;
      props.handleTypes = cudaMemHandleTypeNone;
      props.location.type = cudaMemLocationTypeDevice;
      props.location.id = dev;
      if ((e = cudaMemPoolCreate(&pools[dev], &props)) != cudaSuccess) return e;
      unsigned long long keep = ~0ull;
      if ((e = cudaMemPoolSetAttribute(pools[dev], cudaMemPoolAttrReleaseThreshold, &keep)) != cudaSuccess) return e;
    }
    pool = pools[dev];
    for (int i = 0; i < kStreams; ++i)
      if ((e = cudaStreamCreateWithFlags(&s[i], cudaStreamNonBlocking)) != cudaSuccess) return e;
    return cudaEventCreateWithFlags(&shared_ready, cudaEventDisableTiming);
  }
  // waits for every stream (they may be partly created); the first error
  cudaError_t sync() {
    cudaError_t e = cudaSuccess;
    for (int i = 0; i < kStreams; ++i)
      if (s[i]) {
        const cudaError_t ei = cudaStreamSynchronize(s[i]);
        if (e == cudaSuccess) e = ei;
      }
    return e;
  }
  // frees what init() and alloc() acquired, on every path
  cudaError_t fini() {
    cudaError_t e = sync();
    for (void* p : allocs) cudaFreeAsync(p, s[0]);  // stream 0 owns the allocations; the others are idle now
    allocs.clear();
    if (s[0]) {
      const cudaError_t e0 = cudaStreamSynchronize(s[0]);
      if (e == cudaSuccess) e = e0;
    }
    for (int i = 0; i < kStreams; ++i)
      if (s[i]) { cudaStreamDestroy(s[i]); s[i] = nullptr; }
    if (shared_ready) { cudaEventDestroy(shared_ready); shared_ready = nullptr; }
    return e;
  }

  void* alloc(size_t bytes) {
    void* p = nullptr;
    if (err == cudaSuccess) err = cudaMallocFromPoolAsync(&p, bytes ? bytes : 8, pool, s[0]);
    if (p) allocs.push_back(p);
    return p;
  }
  // register the pointer stored at `slot` of the model (hp: its host value)
  template <class P>
  void add(P* slot, const void* hp, size_t per_member, size_t bytes, unsigned cat) {
    if (!hp) return;
    char* dp = static_cast<char*>(alloc(bytes));
    fields.push_back({(char*)hp, dp, (size_t)((char*)slot - (char*)&d), per_member, bytes, cat});
    *slot = reinterpret_cast<P>(dp);
  }
  void vec(pmoc_vec* dv, long long M, size_t len) {  // input vector: per member when mstride != 0
    if (!dv->ptr) return;
    const size_t stride = (size_t)dv->mstride * sizeof(double);
    const size_t bytes = stride ? (size_t)(M - 1) * stride + len * sizeof(double) : len * sizeof(double);
    add(&dv->ptr, dv->ptr, stride, bytes, kIoParam);
  }
  template <class T>
  void shared(const T** dp, size_t n) { add(dp, *dp, 0, n * sizeof(T), 0); }
  template <class T>
  void state(T** dp, long long M, size_t len, unsigned cat) { add(dp, *dp, len * sizeof(T), (size_t)M * len * sizeof(T), cat); }
  void column(pmoc_column* c, long long M, int nz) {
    state(&c->b, M, nz, PMOC_IO_STATE);
    state(&c->bbot, M, 1, PMOC_IO_STATE);
    state(&c->var, M, 1, PMOC_IO_STATE);
    vec(&c->kappa, M, (size_t)c->nvar * nz);
    vec(&c->dAk, M, (size_t)c->nvar * nz);
    vec(&c->Area, M, nz);
    vec(&c->bs, M, 1);
    vec(&c->N2min, M, 1);
    vec(&c->bzbot, M, 1);
  }
  // register every array of the model, with its class
  void describe() {
    const long long M = d.M;
    const int nz = d.nz, ny = d.ny, nb = d.nb;
    const unsigned f = d.flags;
    const unsigned S = PMOC_IO_STATE, P = PMOC_IO_PSI, D = PMOC_IO_DIAG;
    shared(&d.z, nz);
    shared(&d.y, ny);
    column(&d.basin, M, nz);
    if (f & PMOC_HAS_NORTH) column(&d.north, M, nz);
    if (f & PMOC_HAS_PAC) {
      column(&d.pac, M, nz);
      vec(&d.zoc_f, M, 1);
      vec(&d.so2_L, M, 1);
      state(&d.Psi_zoc, M, nz, D);
      state(&d.Psi_zon_a, M, nz, P);
      state(&d.Psi_zon_p, M, nz, P);
      state(&d.psib2, M, nb, D);
      state(&d.bgrid2, M, nb, D);
      state(&d.Psi_so2, M, nz, P);
      state(&d.Psi_Ek2, M, nz, D);
      state(&d.Psi_GM2, M, nz, D);
    }
    vec(&d.tw_f, M, 1);
    vec(&d.tw_b2, M, nz);
    vec(&d.so_bs, M, ny);
    vec(&d.so_tau, M, d.so_tau_on_y ? ny : 1);
    vec(&d.so_f, M, 1);
    vec(&d.so_rho, M, 1);
    vec(&d.so_L, M, 1);
    vec(&d.so_KGM, M, 1);
    vec(&d.so_smax, M, 1);
    vec(&d.so_c, M, 1);
    shared(&d.so_sill_taper, nz);
    shared(&d.so_ek_taper, nz);
    shared(&d.so_top_taper, nz);
    shared(&d.so_bot_taper, nz);
    state(&d.ml_bs, M, ny, S);
    vec(&d.ml_Ks, M, 1);
    vec(&d.ml_h, M, 1);
    vec(&d.ml_L, M, 1);
    vec(&d.ml_vpist, M, 1);
    vec(&d.ml_surflux, M, ny);
    vec(&d.ml_rest_mask, M, ny);
    vec(&d.ml_b_rest, M, ny);
    state(&d.Psi_tw, M, nz, (f & PMOC_ISO) ? D : P);
    state(&d.Psi_iso_b, M, nz, P);
    state(&d.Psi_iso_n, M, nz, P);
    state(&d.psib, M, nb, D);
    state(&d.bgrid, M, nb, D);
    state(&d.Psi_so, M, nz, P);
    state(&d.Psi_Ek, M, nz, D);
    state(&d.Psi_GM, M, nz, D);
    state(&d.ml_Psi_s, M, ny, D | kIoStepped);
    state(&d.status, M, 1, S);
  }
  // blocks of members: enough of them to overlap copies with kernels, each large enough to fill the GPU; one
  // scratch buffer per stream for the block-per-member kernels (nz > 256)
  long long nblk = 1, per = 0;
  void* scratch[kStreams] = {};
  void plan_blocks() {
    const long long M = d.M;
    nblk = M / PMOC_HOST_BLOCK_MEMBERS;
    if (nblk < 1) nblk = 1;
    if (nblk > 32) nblk = 32;
    per = (M + nblk - 1) / nblk;
    d.scratch = nullptr;
    d.scratch_bytes = 0;
    pmoc_model one = d;
    one.M = per;
    const uint64_t need = pmoc_model_scratch_bytes(&one);
    if (need) {
      for (int i = 0; i < kStreams && i < nblk; ++i) scratch[i] = alloc((size_t)need);
      d.scratch_bytes = need;
    }
  }
  // The shared arrays go up on stream 0 behind the allocations, and the other streams wait for both.
  void upload_shared() {
    for (auto& f : fields)
      if (!f.per_member && err == cudaSuccess) {
        err = cudaMemcpyAsync(f.dev, f.host, f.bytes, cudaMemcpyHostToDevice, s[0]);
        g_h2d_bytes += f.bytes;
      }
    if (err == cudaSuccess) err = cudaEventRecord(shared_ready, s[0]);
    for (int i = 1; i < kStreams && err == cudaSuccess; ++i) err = cudaStreamWaitEvent(s[i], shared_ready, 0);
  }
  // streams, a device copy of every array of `m`, the shared arrays uploaded
  cudaError_t open(const pmoc_model* m) {
    d = *m;
    err = init();
    if (err == cudaSuccess) {
      describe();
      plan_blocks();
    }
    if (err == cudaSuccess) upload_shared();
    return err;
  }

  // Members [m0, m0+n) of the per-member arrays whose class is in `mask`, host->device (`up`) or back, on
  // stream st; the last member of a parameter vector may be shorter than its stride.  With `fill`, the device
  // copy of every other per-member array is zeroed.
  void copy(long long m0, long long n, unsigned mask, bool up, bool fill, cudaStream_t st) {
    for (auto& f : fields) {
      if (!f.per_member || err != cudaSuccess) continue;
      const size_t off = (size_t)m0 * f.per_member, len = std::min((size_t)n * f.per_member, f.bytes - off);
      if (!(f.cat & mask)) {
        if (fill) err = cudaMemsetAsync(f.dev + off, 0, len, st);
      } else if (up) {
        err = cudaMemcpyAsync(f.dev + off, f.host + off, len, cudaMemcpyHostToDevice, st);
        g_h2d_bytes += len;
      } else {
        err = cudaMemcpyAsync(f.host + off, f.dev + off, len, cudaMemcpyDeviceToHost, st);
        g_d2h_bytes += len;
      }
    }
  }
  // the device model restricted to members [m0, m0+n), with the scratch of stream `si`
  pmoc_model block_model(long long m0, long long n, int si) const {
    pmoc_model b = d;
    b.M = n;
    for (auto& f : fields)
      if (f.per_member) *reinterpret_cast<char**>((char*)&b + f.slot) = f.dev + (size_t)m0 * f.per_member;
    b.scratch = scratch[si];
    return b;
  }
  // One call, block by block: the classes in `push` go up (the first upload zeroes every other per-member
  // array), the block is diagnosed (`diag`) and run (`run`), and the classes in `pull` come back.  Returns the
  // first launch error; a CUDA error is left in `err`.
  int pass(unsigned push, bool diag, bool run, long long it0, long long nsteps, unsigned pull) {
    int rc = PMOC_OK;
    for (long long c = 0; c < nblk && rc == PMOC_OK && err == cudaSuccess; ++c) {
      const long long m0 = c * per, n = std::min(per, d.M - m0);
      if (n <= 0) break;
      const int si = (int)(c % kStreams);
      copy(m0, n, push, true, fresh, s[si]);
      pmoc_model blk = block_model(m0, n, si);
      if (diag) rc = pmoc_model_diagnose(&blk, s[si]);
      if (rc == PMOC_OK && run) rc = pmoc_model_run(&blk, it0, nsteps, s[si]);
      if (rc == PMOC_OK) copy(m0, n, pull, false, false, s[si]);
    }
    fresh = false;
    return rc;
  }
};

}  // namespace

extern "C" int pmoc_model_run_host(const pmoc_model* m, int64_t it0, int64_t nsteps) {
  if (!m) return fail(PMOC_EINVAL, "model is NULL");
  g_h2d_bytes = g_d2h_bytes = 0;
  if (m->M <= 0 || m->nz < 3) return fail(PMOC_EINVAL, "bad M / nz");
  // Diagnostics: the kernel rewrites all of them at the last iteration with ii % K == 0 of the launch (and the
  // pre-loop diagnosis of an order-'post' model at it0 == 0 does); without such an iteration they are left
  // alone on both sides.  Only the streamfunctions the step loop carries from an earlier launch are inputs.
  const long long K = m->K > 0 ? m->K : 1;
  const bool jn = (m->flags & PMOC_ORDER_JN) != 0;
  const bool rewritten = (!jn && it0 == 0) || (nsteps > 0 && ((it0 + nsteps - 1) / K) * K >= it0);
  const bool carry = jn ? (it0 % K != 0) : (it0 > 0);
  const unsigned push = kIoParam | PMOC_IO_STATE | (carry ? PMOC_IO_PSI : 0);
  const unsigned pull = PMOC_IO_STATE | (rewritten ? PMOC_IO_PSI | PMOC_IO_DIAG : 0) | (nsteps > 0 ? kIoStepped : 0);
  Mirror mr;
  int rc = PMOC_OK;
  if (mr.open(m) == cudaSuccess) rc = mr.pass(push, !jn && it0 == 0, true, it0, nsteps, pull);
  const cudaError_t e = mr.fini();  // every path: streams, event and device memory are returned
  if (rc != PMOC_OK) return rc;
  PM_CUDA_OK(mr.err);
  PM_CUDA_OK(e);
  return PMOC_OK;
}

// ---- persistent handle: parameters uploaded once, streams and device mirrors kept between calls ------------
struct pmoc_host {
  Mirror mr;
  bool diagnosed = false;
};

extern "C" int pmoc_host_open(const pmoc_model* m, pmoc_host** out) {
  if (!m || !out) return fail(PMOC_EINVAL, "model / handle pointer is NULL");
  *out = nullptr;
  if (m->M <= 0 || m->nz < 3) return fail(PMOC_EINVAL, "bad M / nz");
  pmoc_host* h = new (std::nothrow) pmoc_host();
  if (!h) return fail(PMOC_EINVAL, "out of host memory");
  g_h2d_bytes = g_d2h_bytes = 0;
  Mirror& mr = h->mr;
  // everything goes up once: grids, parameters, state, carried streamfunctions; the diagnostics start at zero
  if (mr.open(m) == cudaSuccess) mr.pass(kIoParam | PMOC_IO_STATE | PMOC_IO_PSI, false, false, 0, 0, 0);
  if (mr.err == cudaSuccess) mr.err = mr.sync();
  if (mr.err != cudaSuccess) {
    const cudaError_t keep = mr.err;
    mr.fini();
    delete h;
    PM_CUDA_OK(keep);
  }
  *out = h;
  return PMOC_OK;
}

extern "C" int pmoc_host_step(pmoc_host* h, int64_t it0, int64_t nsteps, uint32_t push, uint32_t pull) {
  if (!h) return fail(PMOC_EINVAL, "handle is NULL");
  if ((push | pull) & ~(PMOC_IO_STATE | PMOC_IO_PSI | PMOC_IO_DIAG)) return fail(PMOC_EINVAL, "unknown PMOC_IO_* bit");
  if (push & PMOC_IO_DIAG) return fail(PMOC_EINVAL, "diagnostics are outputs: they cannot be pushed");
  g_h2d_bytes = g_d2h_bytes = 0;
  Mirror& mr = h->mr;
  const bool jn = (mr.d.flags & PMOC_ORDER_JN) != 0;
  // an order-'post' loop is entered with diagnosed streamfunctions (the scripts' pre-loop solve()): at it0 == 0,
  // and whenever the caller replaces the state without supplying streamfunctions that match it
  const bool need_diag = !jn && (it0 == 0 || ((push & PMOC_IO_STATE) && !(push & PMOC_IO_PSI) && !h->diagnosed));
  const int rc = mr.pass(push, need_diag, nsteps > 0, it0, nsteps, pull);
  const cudaError_t e = mr.sync();
  if (rc != PMOC_OK) return rc;
  PM_CUDA_OK(mr.err);
  PM_CUDA_OK(e);
  h->diagnosed = true;
  return PMOC_OK;
}

extern "C" int pmoc_host_close(pmoc_host* h) {
  if (!h) return PMOC_OK;
  const cudaError_t e = h->mr.fini();
  delete h;
  PM_CUDA_OK(e);
  return PMOC_OK;
}

// ------------------------------------------------------------------------------------------
#ifdef PMOC_EMU
extern "C" int pmoc_fp64_peak(double*, double*, void*) { return fail(PMOC_ENODEVICE, "the FP64 probe needs a GPU"); }
#else
namespace {
// 8 independent DFMA chains per thread, nothing else: what the FP64 pipe sustains.
__global__ void k_fp64_peak(double* out, int iters, double seed) {
  double a0 = seed + threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6,
         a7 = a0 + 7;
  const double m = 1.0000001, c = 1e-9;
  for (int i = 0; i < iters; ++i) {
    a0 = __fma_rn(a0, m, c); a1 = __fma_rn(a1, m, c); a2 = __fma_rn(a2, m, c); a3 = __fma_rn(a3, m, c);
    a4 = __fma_rn(a4, m, c); a5 = __fma_rn(a5, m, c); a6 = __fma_rn(a6, m, c); a7 = __fma_rn(a7, m, c);
  }
  const double s = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
  if (s == 12345.678) out[0] = s;  // keep the chains alive
}
}  // namespace

extern "C" int pmoc_fp64_peak(double* tflops, double* sm_mhz_est, void* stream) {
  int dev = 0, sms = 0;
  PM_CUDA_OK(cudaGetDevice(&dev));
  PM_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  double* out = nullptr;
  PM_CUDA_OK(cudaMalloc(&out, 8));
  cudaStream_t s = (cudaStream_t)stream;
  cudaEvent_t e0, e1;
  PM_CUDA_OK(cudaEventCreate(&e0));
  PM_CUDA_OK(cudaEventCreate(&e1));
  const int block = 512, grid = sms * 4, iters = 1 << 16;
  k_fp64_peak<<<grid, block, 0, s>>>(out, 2048, 1.0);  // warm-up
  double best = 0.0;
  for (int rep = 0; rep < 5; ++rep) {
    PM_CUDA_OK(cudaEventRecord(e0, s));
    k_fp64_peak<<<grid, block, 0, s>>>(out, iters, 1.0);
    PM_CUDA_OK(cudaEventRecord(e1, s));
    PM_CUDA_OK(cudaEventSynchronize(e1));
    float ms = 0.f;
    PM_CUDA_OK(cudaEventElapsedTime(&ms, e0, e1));
    const double flops = 2.0 * 8.0 * (double)iters * (double)block * (double)grid;
    const double tf = flops / (ms * 1e-3) / 1e12;
    if (tf > best) best = tf;
  }
  PM_CUDA_OK(cudaGetLastError());
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(out);
  if (tflops) *tflops = best;
  // 64 DFMA lanes per SM and clock
  if (sm_mhz_est) *sm_mhz_est = best * 1e12 / (2.0 * 64.0 * sms) / 1e6;
  return PMOC_OK;
}
#endif
