// sm_100a kernels of the GAML assembly-likelihood path. Nothing here is a dense contraction: the work
// is an integer gather over 16-byte alignment records plus a handful of fp64 operations per record, so
// the bound is HBM bandwidth (DESIGN.md §4) and tensor cores are not used.
//
// Exactness contract (DESIGN.md §5): every product/sum that the reference performs in fp64 is issued
// with __dmul_rn/__dadd_rn so no FMA contraction can change a bit; the paired state therefore replays
// ScoringState::probs (graph.cc:1936-1950) bit for bit. Only log/exp/log1p differ from glibc (<= 1-2 ulp).
//
// Execution shape (DESIGN.md §4): one thread per read, reads in id order, so a warp streams 32
// consecutive 16-byte "first" records per mate with one coalesced 512-byte request. Reads with at most
// two live placements per mate (virtually all) are finished in registers; the rest are appended to a
// per-set list and replayed by a second, dense kernel from a scratch arena, so the streaming kernel
// never carries the general sort/de-dup code through its warps.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <type_traits>
#include <utility>

#include "kernels.h"

namespace gaml {

namespace {

constexpr int kCapLong = 8;        // pacbio placements handled in local memory before the scratch path
constexpr int kBlock = 256;
constexpr int kOvfBlock = 128;

// ---- small helpers ------------------------------------------------------------------------
__device__ __forceinline__ int4 ldg4(const void* p) { return __ldg(reinterpret_cast<const int4*>(p)); }
// Streamed-once data: read-only path, not kept in L1 (the lines would only evict the slot and probability tables).
__device__ __forceinline__ uint4 ldg_stream(const uint4* p) {
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}
// PackedPair (16 B per pair, built at cache commit when every record fits): what tier 1 of the streaming kernel needs of
// a pair's two first records — x = key1 | edit1<<22 | orient1<<29 | none1<<30 | tier2<<31, y = the same for mate 2
// (bit 31: both mates under the same key, see apply_slots_kernel), z = pos1, w = pos2. tier2 = some mate owns two or more records (the read is on the static list).
// 256-bit read-only load (sm_100: LDG.E.256): one request, one L1 tag lookup per distinct line for both halves
__device__ __forceinline__ void ldg256(const uint4* p, uint4& a, uint4& b) {
  asm volatile("ld.global.nc.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w), "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w) : "l"(p));
}
constexpr int kPackKeyBits = 22;
constexpr uint32_t kPackKeyMask = (1u << kPackKeyBits) - 1u;
constexpr uint32_t kPackEdMask = 0x7fu;

__device__ __forceinline__ int wrap_add(int a, int b) { return (int)((unsigned)a + (unsigned)b); }

// Programmatic dependent launch (sm_90+): the kernels of one evaluation form a chain on one stream, each launched with
// cudaLaunchAttributeProgrammaticStreamSerialization. pdl_release() lets the NEXT kernel of the chain be launched and
// its blocks become resident while this one still runs; pdl_wait() blocks until the PREVIOUS kernel has completed and
// its writes are visible. Every kernel calls pdl_wait() before it touches anything an earlier kernel of the chain
// wrote (slot words, zeroed flags/accumulators, the overflow list, the read state), so completion is transitive along
// the chain. Both are no-ops for a kernel launched without the attribute.
__device__ __forceinline__ void pdl_release() { asm volatile("griddepcontrol.launch_dependents;"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
// Device timeline (gaml_set_profiling level 2): start of the kernel's first block, end of its last block.
enum { kTlApply = 0, kTlTier1, kTlTier2, kTlOverflow, kTlDelta, kTlTotal, kTlKernels };
__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void tl_begin(unsigned long long* tl, int k) {
  if (tl && threadIdx.x == 0) atomicMax(tl + 2 * k, ~global_ns());   // complemented: the buffer is reset to all zeros
}
__device__ __forceinline__ void tl_end(unsigned long long* tl, int k) {
  if (tl && threadIdx.x == 0) atomicMax(tl + 2 * k + 1, global_ns());
}
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// ---- exact accumulation of the per-read log terms -----------------------------------------------
// Every term is rounded ONCE to a multiple of 2^-40 and added as a 128-bit integer, so the shard total is an
// exact integer sum: associative, hence identical for any grid size, block order, shard count or collective
// order (SURVEY §7.4 item 4). 2^-40 is 6e-15 relative on a typical term of -150; the rounding errors of 2 M terms
// random-walk to ~1e-9 absolute on a total of ~3e8. Non-finite terms (log 0 = -inf, NaN) are counted instead.
constexpr double kFixScale = 1099511627776.0;   // 2^40
constexpr double kFixLimit = 4194304.0;         // |term| < 2^22 so that term * 2^40 fits an int64

struct Acc {
  unsigned long long lo;
  long long hi;
  unsigned neginf, bad;
};
__device__ __forceinline__ Acc acc_zero() { return Acc{0ull, 0ll, 0u, 0u}; }
__device__ __forceinline__ void acc_add_q(Acc& a, long long q) {
  const unsigned long long nlo = a.lo + (unsigned long long)q;
  a.hi += (q >> 63) + (long long)(nlo < (unsigned long long)q);
  a.lo = nlo;
}
__device__ __forceinline__ void acc_count_odd(Acc& a, double lg) {
  if (lg == -INFINITY) a.neginf++;
  else a.bad++;
}
// PacBio terms are log values already (logdouble): rounded once to 2^-40 and added.
__device__ __forceinline__ void acc_add_log(Acc& a, double t) {
  if (fabs(t) < kFixLimit) acc_add_q(a, __double2ll_rn(t * kFixScale));
  else acc_count_odd(a, t);
}

// Block-wide exact sum -> per-set global accumulators {limb0..3 (32-bit limbs in u64), floored, neginf, bad}.
// Warp level: the 128-bit value is cut into eight 16-bit chunks, each summed over the warp by one redux.sync
// (sum < 2^21); block level: the chunk sums meet in shared u32 counters and thread 0 re-assembles them modulo 2^128
// (two's complement, so negatives just work); grid level: four 32-bit limbs by global u64 atomics per block.
// Integer addition commutes, so the atomics do not make the result order dependent.
__device__ void block_accumulate(const Acc& a, unsigned floored, unsigned long long* accum) {
  __shared__ unsigned sm[11];   // eight 16-bit-chunk sums (< 2^21 per warp, < 2^26 per block), floored, -inf, nan
  if (threadIdx.x < 11) sm[threadIdx.x] = 0u;
  __syncthreads();
  const unsigned w[4] = {(unsigned)a.lo, (unsigned)(a.lo >> 32), (unsigned)(unsigned long long)a.hi,
                         (unsigned)((unsigned long long)a.hi >> 32)};
  unsigned s[11];
#pragma unroll
  for (int j = 0; j < 4; j++) {
    s[2 * j] = __reduce_add_sync(0xffffffffu, w[j] & 0xffffu);
    s[2 * j + 1] = __reduce_add_sync(0xffffffffu, w[j] >> 16);
  }
  s[8] = __reduce_add_sync(0xffffffffu, floored);
  s[9] = __reduce_add_sync(0xffffffffu, a.neginf);
  s[10] = __reduce_add_sync(0xffffffffu, a.bad);
  const int lane = threadIdx.x & 31;
  if (lane < 11) {   // lane j publishes chunk j: one shared atomic per lane instead of a 128-bit re-assembly per warp
    unsigned v = s[0];
#pragma unroll
    for (int j = 1; j < 11; j++) v = lane == j ? s[j] : v;
    if (v) atomicAdd(&sm[lane], v);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned __int128 x = 0;   // sum of chunk_j << 16j modulo 2^128 (two's complement: negatives just work)
#pragma unroll
    for (int j = 0; j < 8; j++) x += (unsigned __int128)sm[j] << (16 * j);
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const unsigned long long limb = (unsigned long long)(unsigned)(x >> (32 * j));
      if (limb) atomicAdd(accum + j, limb);
    }
    // counters may be net negative in a delta-only evaluation: sign-extend (the 64-bit sums are modulo 2^64)
    if (sm[8]) atomicAdd(accum + 4, (unsigned long long)(long long)(int)sm[8]);
    if (sm[9]) atomicAdd(accum + 5, (unsigned long long)(long long)(int)sm[9]);
    if (sm[10]) atomicAdd(accum + 6, (unsigned long long)(long long)(int)sm[10]);
  }
}

// Thread 0 of the block that completes a read set: re-assembles the set's exact 128-bit sum from its limbs and writes
// out[] = {integer part, fraction in 2^-40 units, floored, -inf terms, nan terms, flags} (both parts are integers
// below 2^53, exact in a double) straight into the host's result buffer (zero-copy), followed by the evaluation's
// epoch as the completion flag. Out of line and fed by value: it runs once per evaluation, and a reference to the
// kernel's parameter block would force a local copy of all of it in every thread of the streaming kernels.
struct PublishArgs {
  const unsigned long long* accum;
  unsigned long long* state_acc;
  double* out;
  const uint32_t* error_flag;
  const uint32_t* ovf_count;
  const unsigned long long* scratch_cursor;
  uint32_t* ticket;
  uint32_t* done;
  uint32_t epoch;
  int32_t state_add;
  long long ql;        // FIX(log 2L): subtracted once per read whose term is a logarithm of its value (0 for PacBio sets)
  long long n_reads;
  unsigned long long* const* peer_bufs;   // multi-GPU: every rank's exchange buffer (peer memory), or null
  int32_t peer_world;
  uint32_t peer_line;
  double* part_out;
  int32_t last_in_chain;   // the streaming kernel ends the chain (finish_here 2): listed reads give a pending line
};
__device__ __forceinline__ PublishArgs publish_args(const ScoreParams& P, uint32_t* ticket) {
  return PublishArgs{P.accum, P.state_acc, P.out, P.error_flag, P.ovf_count, P.scratch_cursor, ticket, P.done, P.epoch, P.state_add,
                     P.ql, (long long)P.n_reads, P.peer_bufs, P.peer_world, P.peer_line, P.part_out, P.finish_here == 2};
}

// Called by the first warp of the completing block. Lane 0 assembles the eight result words; lanes 0..7 then store
// one word each with ONE instruction — a single 64-byte write to the host instead of eight, and no system-wide fence
// between payload and flag: word 6 is the evaluation's epoch (the flag the host spins on) and word 7 a checksum of
// the other seven, so the host accepts the line only when it is complete, whatever order its bytes arrive in.
// pending: the set still owes the terms of the reads listed for the many-placement pass, which the owning host runs
// on demand. Word 6 is then -epoch, which no host waiting for the final line accepts, and the running total is left
// alone (that pass commits it).
__device__ __noinline__ void publish_set(PublishArgs A, bool pending) {
  const int lane = threadIdx.x & 31;
  unsigned long long w[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (lane == 0) {
    __threadfence();
    unsigned long long a[7];
    for (int j = 0; j < 7; j++) a[j] = __ldcg(A.accum + j);
    unsigned __int128 x = 0;
    for (int j = 0; j < 4; j++) x += (unsigned __int128)a[j] << (32 * j);
    if (A.state_acc && !pending) {
      // paired sets keep their running total {low, high 64 bits, floored, -inf, nan} on the device: a delta-only
      // evaluation accumulated (new term - old term) of the touched reads and adds it, any other sets it
      if (A.state_add) {
        x += ((unsigned __int128)__ldcg(A.state_acc + 1) << 64) | (unsigned __int128)__ldcg(A.state_acc);
        for (int j = 4; j < 7; j++) a[j] += __ldcg(A.state_acc + j - 2);
      }
      A.state_acc[0] = (unsigned long long)x;
      A.state_acc[1] = (unsigned long long)(x >> 64);
      for (int j = 4; j < 7; j++) A.state_acc[j - 2] = a[j];
    }
    // every read contributes exactly one term; those that are neither floored nor non-finite are FIX(LOG p) and still owe
    // their - FIX(log 2L) (see acc_term): one exact integer product
    const long long n_log = A.n_reads - (long long)a[4] - (long long)a[5] - (long long)a[6];
    const __int128 v = (__int128)x - (__int128)n_log * (__int128)A.ql;
    const unsigned __int128 xv = (unsigned __int128)v;
    const unsigned long long scratch = __ldcg(A.scratch_cursor);   // placements parked in the scratch arena
    w[0] = (unsigned long long)__double_as_longlong((double)(long long)(v >> 40));
    w[1] = (unsigned long long)__double_as_longlong((double)(unsigned long long)(xv & (((unsigned __int128)1 << 40) - 1)));
    w[2] = (unsigned long long)__double_as_longlong((double)a[4]);
    w[3] = (unsigned long long)__double_as_longlong((double)a[5]);
    w[4] = (unsigned long long)__double_as_longlong((double)a[6]);
    // flags: error bits (4) | listed reads (24 bits) | scratch placements (24 bits, saturating)
    w[5] = (unsigned long long)__double_as_longlong((double)__ldcg(A.error_flag) + 16.0 * (double)min(__ldcg(A.ovf_count), 0xffffffu) +
                                                    268435456.0 * (double)min(scratch, 0xffffffull));
    w[6] = (unsigned long long)__double_as_longlong(pending ? -(double)A.epoch : (double)A.epoch);
    w[7] = kResultSeal;
    for (int j = 0; j < 7; j++) w[7] ^= w[j];
  }
  unsigned long long mine = 0;
#pragma unroll
  for (int j = 0; j < 8; j++) {
    const unsigned long long v = __shfl_sync(0xffffffffu, w[j], 0);
    if (lane == j) mine = v;
  }
  if (lane < 8) reinterpret_cast<unsigned long long*>(A.out)[lane] = mine;
  if (A.part_out && lane < 8) reinterpret_cast<unsigned long long*>(A.part_out)[lane] = mine;
  if (A.peer_bufs) {
    // the all-gather of a multi-GPU evaluation, fused into the kernel: one 64-byte store per rank over NVLink peer
    // memory. The line validates itself (epoch + checksum), so no flag, fence or ordering is needed on this side.
    for (int p = 0; p < A.peer_world; p++) {
      unsigned long long* dst = A.peer_bufs[p] + (size_t)A.peer_line * kResultStride;
      if (lane < 8) dst[lane] = mine;
    }
    __threadfence_system();
  }
}

// Last kernel of a multi-GPU evaluation's chain (one block): waits until the lines of ALL ranks for this evaluation have
// arrived in this rank's exchange buffer — each thread polls one (rank, set) line until its epoch word and checksum are
// right — copies them to the host-mapped gather area and then writes one flag line the host spins on. A peer that never
// publishes (it died, or the ranks fell out of lockstep) is given `timeout_ns`; the flag line then carries status 1.
__global__ void __launch_bounds__(kResultStride * 32) exchange_gather_kernel(const unsigned long long* lines, int world, int n_sets, int max_sets,
                                                                              uint32_t epoch, unsigned long long* host_lines,
                                                                              unsigned long long* host_flag, unsigned long long timeout_ns) {
  pdl_release();
  __shared__ int s_fail;
  if (threadIdx.x == 0) s_fail = 0;
  __syncthreads();
  const unsigned long long want = (unsigned long long)__double_as_longlong((double)epoch);
  const unsigned long long t0 = global_ns();
  for (int i = threadIdx.x; i < world * n_sets; i += blockDim.x) {
    const int rk = i / n_sets, st = i % n_sets;
    const volatile unsigned long long* src = lines + ((size_t)rk * max_sets + st) * kResultStride;
    unsigned long long w[8];
    for (;;) {
#pragma unroll
      for (int j = 0; j < 8; j++) w[j] = src[j];
      unsigned long long sum = kResultSeal;
#pragma unroll
      for (int j = 0; j < 7; j++) sum ^= w[j];
      if (w[6] == want && w[7] == sum) break;
      if (global_ns() - t0 > timeout_ns) {
        s_fail = 1;
        break;
      }
    }
    unsigned long long* dst = host_lines + (size_t)i * kResultStride;
#pragma unroll
    for (int j = 0; j < 8; j++) dst[j] = w[j];
  }
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x < 8) {
    unsigned long long w[8] = {(unsigned long long)s_fail, 0, 0, 0, 0, 0, want, kResultSeal};
    for (int j = 0; j < 7; j++) w[7] ^= w[j];
    host_flag[threadIdx.x] = w[threadIdx.x];
  }
}

// After a collective library's all-reduce of the ranks' lines (sums of doubles: exact, every field is an integer far
// below 2^53): rebuild one valid line per set — summed partials, this evaluation's epoch, checksum — in host-mapped memory.
__global__ void reduced_publish_kernel(const double* reduced, int n_sets, uint32_t epoch, unsigned long long* host_lines) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_sets) return;
  unsigned long long w[8];
  for (int j = 0; j < 6; j++) w[j] = (unsigned long long)__double_as_longlong(reduced[(size_t)s * kResultStride + j]);
  w[6] = (unsigned long long)__double_as_longlong((double)epoch);
  w[7] = kResultSeal;
  for (int j = 0; j < 7; j++) w[7] ^= w[j];
  __threadfence_system();
  for (int j = 0; j < 8; j++) host_lines[(size_t)s * kResultStride + j] = w[j];
}

// Block-level tail of a set's kernels. early = false: called by every block of the set's LAST kernel, the block that
// draws the final ticket publishes. early = true: called by every block of the set's last STREAMING kernel
// (P.finish_here): if no read was listed for the many-placement pass, the last block publishes right away and marks the
// set done — the pass that follows in the chain then has nothing to do, and the host has its result one kernel earlier.
// When no pass follows (A.last_in_chain) and reads were listed, the last block publishes a pending line instead: the
// owning host then runs the many-placement pass, which publishes the final one.
__device__ __noinline__ void finish_blocks(PublishArgs A, bool early) {
  __shared__ bool s_last, s_pending;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    bool last = atomicAdd(A.ticket, 1u) == gridDim.x - 1;
    bool pending = false;
    if (last && early) {
      __threadfence();
      pending = __ldcg(A.ovf_count) != 0;
      last = !pending || A.last_in_chain;
    }
    s_last = last;
    s_pending = pending;
  }
  __syncthreads();
  if (!s_last || threadIdx.x >= 32) return;
  const bool pending = s_pending;
  publish_set(A, pending);
  if (early && !pending && threadIdx.x == 0) *A.done = 1u;
}
__device__ __forceinline__ void finish_set(const ScoreParams& P) { finish_blocks(publish_args(P, P.ticket2), false); }
__device__ __forceinline__ void finish_set_if_complete(const ScoreParams& P) { finish_blocks(publish_args(P, P.ticket), true); }

// ---- log and division ------------------------------------------------------------------------------
// log(v) for positive normal finite v from a 128-entry table {1/c, -log(1/c)} (host-built in long double,
// engine.cu): v = 2^k z, z in [0.6875, 1.375); r = z*invc - 1 (one fma, |r| < 2^-7); log v = k ln2 + logc + log1p(r)
// with a degree-7 Taylor polynomial (truncation < 2e-19). About 1 ulp; everything else falls back to log().
// Rare paths kept out of line so the compiler cannot if-convert them into the hot loops (ncu showed the IEEE
// division being issued, predicated off, on every iteration when it was inline).
__device__ __noinline__ double slow_log(double v) { return log(v); }

__device__ __forceinline__ double table_log(const double2* __restrict__ tab, double v) {
  const long long ix = __double_as_longlong(v);
  if ((unsigned long long)(ix - 0x0010000000000000ll) >= 0x7fe0000000000000ull) return slow_log(v);   // 0, denormal, inf, nan, < 0
  const long long tmp = ix - 0x3fe6000000000000ll;
  const int i = (int)((tmp >> 45) & 127);
  const long long k = tmp >> 52;
  const double z = __longlong_as_double(ix - (tmp & 0xfff0000000000000ll));
  const double2 e = tab[i];
  const double r = fma(z, e.x, -1.0);
  double p = fma(r, 1.0 / 7.0, -1.0 / 6.0);
  p = fma(r, p, 0.2);
  p = fma(r, p, -0.25);
  p = fma(r, p, 1.0 / 3.0);
  p = fma(r, p, -0.5);
  p = fma(r * r, p, r);
  return fma((double)k, 0.693147180559945309417232121458, e.y) + p;
}

// The per-read log term of GetTotalProb (graph.cc:1495-1537): log max(p / 2L, thr), restated so that nothing in it
// needs a division or depends on L except one comparison:
//   floored  <=>  RN(p / 2L) < thr  <=>  p < pstar, pstar = the smallest double whose IEEE quotient by 2L reaches thr
//                 (found on the host per evaluation and read length: the decision is EXACTLY the reference's);
//   floored:   FIX(log thr)                 (host table, glibc log of the reference's own threshold)
//   otherwise: FIX(LOG p) - FIX(log 2L)     (log(p / 2L) = log p - log 2L to ~1e-14 absolute, far inside the 1e-12 per-read
//                 bar; FIX = rounded once to 2^-40). Only the first part is accumulated here; the block that publishes a
//                 set subtracts (number of such reads) * FIX(log 2L) from the exact integer sum (publish_set).
// LOG p depends on the read's value alone, so it can be tabulated next to the pair term (TermEntry), and every kernel —
// streaming, delta, total, many-placement, batch — forms bit-identical integers for the same value, which is what lets
// the running total swap a read's old term for its new one.
__device__ __forceinline__ void acc_term(Acc& a, unsigned& floored, const double2* log_tab, double p, double pstar, long long qthr) {
  if (p < pstar) {
    floored++;
    acc_add_q(a, qthr);
    return;
  }
  const double lg = table_log(log_tab, p);
  if (fabs(lg) < kFixLimit) acc_add_q(a, __double2ll_rn(lg * kFixScale));
  else acc_count_odd(a, lg);
}
// Removes a term an EARLIER evaluation added for the same value at the same total length (same pstar): the running total
// of a paired set is updated in O(touched reads). The counters wrap modulo 2^32 and are sign-extended in block_accumulate.
__device__ __forceinline__ void acc_term_sub(Acc& a, unsigned& floored, const double2* log_tab, double p, double pstar, long long qthr) {
  if (p < pstar) {
    floored--;
    acc_add_q(a, -qthr);
    return;
  }
  const double lg = table_log(log_tab, p);
  if (fabs(lg) < kFixLimit) acc_add_q(a, -__double2ll_rn(lg * kFixScale));
  else if (lg == -INFINITY) a.neginf--;
  else a.bad--;
}
// Floor test and floored term of a read with packed lengths ll (paired) or length ll (single).
__device__ __forceinline__ void term_consts(const ScoreParams& P, uint32_t len_index, double& pstar, long long& qthr) {
  pstar = __ldg(P.pstar_tab + len_index);
  qthr = __ldg(P.qthr_tab + len_index);
}
__device__ __forceinline__ void acc_read(const ScoreParams& P, Acc& a, unsigned& floored, double p, uint32_t len_index) {
  double pstar;
  long long qthr;
  term_consts(P, len_index, pstar, qthr);
  acc_term(a, floored, static_cast<const double2*>(P.log_tab), p, pstar, qthr);
}
// the fixed-point logarithm of a value for the term tables: kTermOdd when it is not finite
__device__ __forceinline__ long long fix_log(const double2* log_tab, double p) {
  const double lg = table_log(log_tab, p);
  return fabs(lg) < kFixLimit ? __double2ll_rn(lg * kFixScale) : kTermOdd;
}

// ---- placement enumeration ----------------------------------------------------------------
// One live key occurrence applied to one record: F(occurrence int4 {walk, seg, cur_pos, skip_below}, row, row index).
template <class F>
__device__ __forceinline__ void visit_row(const MateView& mv, uint32_t epoch, const int4& rw, int idx, F&& f) {
  const int4 a = ldg4(mv.slots_a + rw.x);                     // {epoch | multi<<31, walk, cur_pos, skip_below}
  if (((uint32_t)a.x & 0x7fffffffu) != epoch) return;
  const int4 b = ldg4(mv.slots_b + rw.x);                     // {seg, n_occ, occ_begin, -}
  f(make_int4(a.y, b.x, a.z, a.w), rw, idx);
  for (int t = 1; t < b.y; t++) f(ldg4(mv.occ + b.z + t), rw, idx);
}

// Candidate-local key table of a batched evaluation (gaml_calc_prob_batch): the few keys of the walks one candidate
// move erases/adds, sorted by key id, with the same two slot words. Found by binary search instead of the global
// epoch-stamped table, so 1024 candidates with different walk sets can be scored in one launch.
struct CandLookup {
  const int* keys;
  int n;
  const int4* a;
  const int4* b;
  const Occ* occ;
};
template <class F>
__device__ __forceinline__ void visit_row(const MateView&, const CandLookup& lk, const int4& rw, int idx, F&& f) {
  int lo = 0, hi = lk.n;   // (plain loads: the tables may sit in shared memory — batch_touch_kernel stages them)
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (lk.keys[mid] < rw.x) lo = mid + 1; else hi = mid;
  }
  if (lo >= lk.n || lk.keys[lo] != rw.x) return;
  const int4 a = lk.a[lo], b = lk.b[lo];
  f(make_int4(a.y, b.x, a.z, a.w), rw, idx);
  for (int t = 1; t < b.y; t++) f(ldg4(lk.occ + b.z + t), rw, idx);
}

// Short-read stores (hybrid layout): first[r] = {key, pos, edor | count<<16, row offset}; the read's
// other records follow at rows[offset+1 ..]. key < 0 = the read has no record at all.
template <class E, class F>
__device__ __forceinline__ void for_each_short(const MateView& mv, const E& epoch, int r, F&& f) {
  int4 rw = ldg4(static_cast<const int4*>(mv.first) + r);
  if (rw.x < 0) return;
  int cnt = (rw.z >> 16) & 0x3fff;
  const uint32_t base = (uint32_t)rw.w;
  if (cnt == 0x3fff) cnt = (int)(__ldg(mv.rowptr + r + 1) - base);
  rw.z &= 0x4000ffff;
  visit_row(mv, epoch, rw, 0, f);
  const RowShort* rows = static_cast<const RowShort*>(mv.rows);
  for (int i = 1; i < cnt; i++) visit_row(mv, epoch, ldg4(rows + base + i), i, f);
}

// Compact copy of the records of the tier-2 reads (those owning several records on a mate): read k of the
// static list owns crows[cptr[k] .. cptr[k+1]) — contiguous across neighbouring threads, so tier 2 streams.
template <class E, class F>
__device__ __forceinline__ void for_each_compact(const MateView& mv, const E& epoch, int k, F&& f) {
  const uint32_t b = __ldg(mv.cptr + k), e = __ldg(mv.cptr + k + 1);
  const RowShort* rows = static_cast<const RowShort*>(mv.crows);
  for (uint32_t i = b; i < e; i++) visit_row(mv, epoch, ldg4(rows + i), (int)(i - b), f);
}

// PacBio stores: plain CSR.
template <class F>
__device__ __forceinline__ void for_each_long(const MateView& mv, uint32_t epoch, int r, F&& f) {
  const uint32_t b = __ldg(mv.rowptr + r), e = __ldg(mv.rowptr + r + 1);
  const RowLong* rows = static_cast<const RowLong*>(mv.rows);
  for (uint32_t i = b; i < e; i++) visit_row(mv, epoch, ldg4(rows + i), (int)(i - b), f);
}

template <class T>
__device__ __forceinline__ void sort_by_ord(T* p, int n) {
  for (int i = 1; i < n; i++) {
    T v = p[i];
    int j = i - 1;
    while (j >= 0 && p[j].ord > v.ord) { p[j + 1] = p[j]; j--; }
    p[j + 1] = v;
  }
}

// De-duplicate [b,e) in place by position: first occurrence keeps the slot, a later record with the
// same position overwrites its payload (graph.cc:583-592, 635-641). Returns the new end.
__device__ __forceinline__ int dedup_positions(Plc* p, int b, int e) {
  int out = b;
  for (int k = b; k < e; k++) {
    int t = b;
    for (; t < out; t++)
      if (p[t].pos == p[k].pos) break;
    if (t < out) p[t].edor = p[k].edor;
    else p[out++] = p[k];
  }
  return out;
}

// ---- paired -------------------------------------------------------------------------------
__device__ __forceinline__ double align_prob(const MateView& mv, int edor, int len) {
  const int ed = edor & 0xffff;
  return __dmul_rn(__ldg(mv.pow_mismatch + ed), __ldg(mv.pow_match + (len - ed)));   // graph.cc:1859-1863
}

// One (x, y) combination of graph.cc:1861-1889; returns false when the orientation/order filter drops it.
// Coverage-gap penalty input (graph.cc:1883-1888): a pair whose term exceeds exp(mps + mppb*2*len2) marks both of
// its positions as "covered" in its walk. Events are appended as sortable keys walk<<33 | (pos ^ 2^31)<<1 | 1.
__device__ __forceinline__ unsigned long long cov_key(int walk, int pos, int type3) {
  return ((unsigned long long)(uint32_t)walk << 33) | ((unsigned long long)((uint32_t)pos ^ 0x80000000u) << 1) |
         (unsigned long long)type3;
}
__device__ __forceinline__ void emit_cov(const ScoreParams& P, int walk, int xpos, int ypos, int l2, double term) {
  if (!P.ev_keys || walk < 0 || !(term > __ldg(P.cov_thr + l2))) return;
  const unsigned i = atomicAdd(P.ev_count, 2u);
  if (i + 2u > P.ev_cap) {
    atomicOr(P.error_flag, 4u);
    return;
  }
  P.ev_keys[i] = cov_key(walk, max(xpos, ypos), 1);
  P.ev_keys[i + 1] = cov_key(walk, min(xpos, ypos), 1);   // use_all_to_cov is always true here (prob_calculator.h:93)
}

__device__ __forceinline__ bool pair_term(const ScoreParams& P, int walk, int xpos, int xedor, int ypos, int yedor, int l1,
                                          int l2, double p1, double& term) {
  const int xo = (xedor >> 30) & 1, yo = (yedor >> 30) & 1;
  if (xo == yo) return false;
  int d;
  if (xpos < ypos) {
    if (xo != 0) return false;
    d = ypos - xpos + l2;
  } else {
    if (xo != 1) return false;
    d = xpos - ypos + l1;
  }
  const double p2 = align_prob(P.m[1], yedor, l2);
  const double ins = ((unsigned)d < (unsigned)P.ins_n) ? __ldg(P.ins_tab + d) : 0.0;
  term = __dmul_rn(__dmul_rn(p1, p2), ins);
  emit_cov(P, walk, xpos, ypos, l2, term);
  return true;
}

// Up to kFew placements of one mate, in registers (every index below is a compile-time constant after unrolling).
// An incremental evaluation doubles a read's placements — the same record sits on the erased walk and on the added
// one — so four covers what two covers in a full evaluation.
constexpr int kFew = 4;
struct Few {
  int n;
  unsigned long long ord[kFew];
  int walk[kFew], pos[kFew], edor[kFew];
};
using Two = Few;   // (single-read path and older call sites)

template <bool kCompact = false, class E = uint32_t>
__device__ __forceinline__ void scan_two(const MateView& mv, const E& epoch, int r, Few& t) {
  t.n = 0;
  auto visit = [&](const int4& o, const int4& rw, int idx) {
    const int pos = wrap_add(rw.y, o.z);
    if (pos < o.w) return;   // graph.cc:577
    const unsigned long long ord = ((unsigned long long)(uint32_t)o.y << 32) | (uint32_t)idx;
#pragma unroll
    for (int j = 0; j < kFew; j++)
      if (t.n == j) { t.ord[j] = ord; t.walk[j] = o.x; t.pos[j] = pos; t.edor[j] = rw.z; }
    t.n++;
  };
  if (kCompact) for_each_compact(mv, epoch, r, visit);
  else for_each_short(mv, epoch, r, visit);
}

__device__ __forceinline__ void few_swap(Few& t, int i, int j) {
  const unsigned long long o = t.ord[i]; t.ord[i] = t.ord[j]; t.ord[j] = o;
  int x;
  x = t.walk[i]; t.walk[i] = t.walk[j]; t.walk[j] = x;
  x = t.pos[i]; t.pos[i] = t.pos[j]; t.pos[j] = x;
  x = t.edor[i]; t.edor[i] = t.edor[j]; t.edor[j] = x;
}

// Enumeration order (sorting network; absent entries get the largest key) + per-walk de-dup: the first occurrence of
// a (walk, position) keeps its slot, a later one overwrites its payload and disappears (graph.cc:583-592).
// Returns a validity mask over the kFew slots.
__device__ __forceinline__ unsigned order_few(Few& t) {
#pragma unroll
  for (int j = 0; j < kFew; j++)
    if (j >= t.n) t.ord[j] = ~0ull;
#define GAML_CSWAP(I, J) if (t.ord[J] < t.ord[I]) few_swap(t, I, J);
  GAML_CSWAP(0, 1) GAML_CSWAP(2, 3) GAML_CSWAP(0, 2) GAML_CSWAP(1, 3) GAML_CSWAP(1, 2)
#undef GAML_CSWAP
  unsigned valid = (1u << t.n) - 1u;
#pragma unroll
  for (int j = 1; j < kFew; j++) {
    bool merged = false;
#pragma unroll
    for (int i = 0; i < j; i++) {
      if (!merged && ((valid >> i) & 1u) && ((valid >> j) & 1u) && t.walk[i] == t.walk[j] && t.pos[i] == t.pos[j]) {
        t.edor[i] = t.edor[j];
        valid &= ~(1u << j);
        merged = true;
      }
    }
  }
  return valid;
}

__device__ __forceinline__ void one_pair(const ScoreParams& P, int xw, int xp, int xe, int yw, int yp, int ye, int l1,
                                         int l2, double p1, double& acc, int n_erased) {
  if (xw != yw) return;
  double t;
  if (pair_term(P, xw, xp, xe, yp, ye, l1, l2, p1, t)) acc = (xw < n_erased) ? __dsub_rn(acc, t) : __dadd_rn(acc, t);
}

// Per-read paired update for reads with <= kFew live placements per mate. For lists sorted in enumeration
// order the plain x-major / y-minor loop with a same-walk filter IS the reference's order: walks ascend with
// x, erased walks (subtract) precede added ones (add). Returns false if the read needs the scratch path.
template <bool kCompact = false, class E0 = uint32_t, class E1 = uint32_t>
__device__ __forceinline__ bool paired_read_with(const ScoreParams& P, const E0& lk0, const E1& lk1, int r, double& acc, int n_erased) {
  Few a, b;
  const uint32_t ll = __ldg((kCompact ? P.clens : P.lens) + r);   // r is the list index k in the compact variant
  scan_two<kCompact>(P.m[0], lk0, r, a);
  if (a.n == 0) return true;
  scan_two<kCompact>(P.m[1], lk1, r, b);
  if (b.n == 0) return true;
  if (a.n > kFew || b.n > kFew) return false;
  const int l1 = ll & 0xffff, l2 = ll >> 16;
  const unsigned va = order_few(a), vb = order_few(b);
#pragma unroll
  for (int x = 0; x < kFew; x++) {
    if (!((va >> x) & 1u)) continue;
    const double p1 = align_prob(P.m[0], a.edor[x], l1);
#pragma unroll
    for (int y = 0; y < kFew; y++)
      if ((vb >> y) & 1u) one_pair(P, a.walk[x], a.pos[x], a.edor[x], b.walk[y], b.pos[y], b.edor[y], l1, l2, p1, acc, n_erased);
  }
  return true;
}

template <bool kCompact = false>
__device__ __forceinline__ bool paired_read(const ScoreParams& P, int r, double& acc) {
  return paired_read_with<kCompact>(P, P.epoch, P.epoch, r, acc, P.n_erased);
}

// Level-batched form of paired_read for the shapes the ordered paths mostly see (incremental evaluations, where a
// record's key is usually live twice — on the erased walk and on the added one — and the multi / many-placement
// passes). paired_read walks one dependent load after
// another (first record -> slot A -> slot B -> further occurrences -> next row ...) per mate; these kernels run one
// read per thread, so that chain IS their run time. Here everything at the same depth is issued together for both
// mates: {first records, lengths} -> {the other rows} -> {both slot words of every row} -> {second occurrences}.
// Covers up to four records per mate, keys occurring at most twice, at most four live placements per mate.
// Returns 1 = scored, -1 = shape not covered.
__device__ __forceinline__ void few_push(Few& t, int walk, int seg, int cur, int skip, const int4& rw, int idx) {
  const int pos = wrap_add(rw.y, cur);
  if (pos < skip) return;   // graph.cc:577
  const unsigned long long ord = ((unsigned long long)(uint32_t)seg << 32) | (uint32_t)idx;
#pragma unroll
  for (int j = 0; j < kFew; j++)
    if (t.n == j) { t.ord[j] = ord; t.walk[j] = walk; t.pos[j] = pos; t.edor[j] = rw.z; }
  t.n++;
}

constexpr int kBatchRec = 4;   // records per mate the level-batched path loads (absent ones are predicated off)

__device__ __forceinline__ int paired_read_fast(const ScoreParams& P, int r, double& acc) {
  int4 rw[2][kBatchRec], sa[2][kBatchRec], sb[2][kBatchRec], oc[2][kBatchRec];
  int cnt[2];
  rw[0][0] = ldg4(static_cast<const int4*>(P.m[0].first) + r);
  rw[1][0] = ldg4(static_cast<const int4*>(P.m[1].first) + r);
  const uint32_t ll = __ldg(P.lens + r);
  if (rw[0][0].x < 0 || rw[1][0].x < 0) return 1;   // a mate without any record: no pair term can exist
  cnt[0] = (rw[0][0].z >> 16) & 0x3fff;
  cnt[1] = (rw[1][0].z >> 16) & 0x3fff;
  if (cnt[0] > kBatchRec || cnt[1] > kBatchRec) return -1;
  // level 2: the other rows
#pragma unroll
  for (int m = 0; m < 2; m++) {
    const RowShort* rows = static_cast<const RowShort*>(P.m[m].rows) + (uint32_t)rw[m][0].w;
#pragma unroll
    for (int i = 1; i < kBatchRec; i++) rw[m][i] = i < cnt[m] ? ldg4(rows + i) : rw[m][0];
    rw[m][0].z &= 0x4000ffff;
  }
  // level 3: both slot words of every row (an absent row repeats the first row's key: same cache line)
#pragma unroll
  for (int m = 0; m < 2; m++)
#pragma unroll
    for (int i = 0; i < kBatchRec; i++) {
      sa[m][i] = ldg4(P.m[m].slots_a + rw[m][i].x);
      sb[m][i] = ldg4(P.m[m].slots_b + rw[m][i].x);
    }
  const uint32_t e = P.epoch;
  bool live[2][kBatchRec];
  bool too_many = false;
#pragma unroll
  for (int m = 0; m < 2; m++)
#pragma unroll
    for (int i = 0; i < kBatchRec; i++) {
      live[m][i] = i < cnt[m] && ((uint32_t)sa[m][i].x & 0x7fffffffu) == e;
      too_many |= live[m][i] && sb[m][i].y > 2;
    }
  if (too_many) return -1;
  // level 4: the second occurrence of the keys that have one
#pragma unroll
  for (int m = 0; m < 2; m++)
#pragma unroll
    for (int i = 0; i < kBatchRec; i++)
      oc[m][i] = (live[m][i] && sb[m][i].y == 2) ? ldg4(P.m[m].occ + sb[m][i].z + 1) : make_int4(0, 0, 0, 0);
  Few t[2];
#pragma unroll
  for (int m = 0; m < 2; m++) {
    t[m].n = 0;
#pragma unroll
    for (int i = 0; i < kBatchRec; i++) {
      if (!live[m][i]) continue;
      few_push(t[m], sa[m][i].y, sb[m][i].x, sa[m][i].z, sa[m][i].w, rw[m][i], i);
      if (sb[m][i].y == 2) few_push(t[m], oc[m][i].x, oc[m][i].y, oc[m][i].z, oc[m][i].w, rw[m][i], i);
    }
  }
  if (t[0].n == 0 || t[1].n == 0) return 1;
  if (t[0].n > kFew || t[1].n > kFew) return -1;
  const int l1 = ll & 0xffff, l2 = ll >> 16;
  const unsigned va = order_few(t[0]), vb = order_few(t[1]);
#pragma unroll
  for (int x = 0; x < kFew; x++) {
    if (!((va >> x) & 1u)) continue;
    const double p1 = align_prob(P.m[0], t[0].edor[x], l1);
#pragma unroll
    for (int y = 0; y < kFew; y++)
      if ((vb >> y) & 1u)
        one_pair(P, t[0].walk[x], t[0].pos[x], t[0].edor[x], t[1].walk[y], t[1].pos[y], t[1].edor[y], l1, l2, p1, acc, P.n_erased);
  }
  return 1;
}

// The ordered register paths in turn: level-batched shapes first, then the general walk; false = scratch path.
__device__ __forceinline__ bool paired_read_ordered(const ScoreParams& P, int r, double& acc) {
  const int st = paired_read_fast(P, r, acc);
  if (st > 0) return true;
  return paired_read(P, r, acc);
}

// General replay from placement lists in memory (scratch path).
template <class E>
__device__ int gather_short(const MateView& mv, const E& epoch, int r, Plc* out) {
  int n = 0;
  for_each_short(mv, epoch, r, [&](const int4& o, const int4& rw, int idx) {
    const int pos = wrap_add(rw.y, o.z);
    if (pos < o.w) return;
    if (out) {
      Plc p;
      p.ord = ((unsigned long long)(uint32_t)o.y << 32) | (uint32_t)idx;
      p.walk = o.x;
      p.pos = pos;
      p.edor = rw.z;
      p.pad = 0;
      out[n] = p;
    }
    n++;
  });
  return n;
}

__device__ double apply_pairs(const ScoreParams& P, Plc* a, int n1, Plc* b, int n2, int l1, int l2, double acc, int n_erased) {
  sort_by_ord(a, n1);
  sort_by_ord(b, n2);
  // per-walk de-dup (lists are walk-major after the sort)
  int m1 = 0, m2 = 0;
  for (int i = 0; i < n1;) {
    int e = i;
    while (e < n1 && a[e].walk == a[i].walk) e++;
    const int end = dedup_positions(a, i, e);
    for (int k = i; k < end; k++) a[m1++] = a[k];
    i = e;
  }
  for (int i = 0; i < n2;) {
    int e = i;
    while (e < n2 && b[e].walk == b[i].walk) e++;
    const int end = dedup_positions(b, i, e);
    for (int k = i; k < end; k++) b[m2++] = b[k];
    i = e;
  }
  for (int x = 0; x < m1; x++) {
    const double p1 = align_prob(P.m[0], a[x].edor, l1);
    for (int y = 0; y < m2; y++) one_pair(P, a[x].walk, a[x].pos, a[x].edor, b[y].walk, b[y].pos, b[y].edor, l1, l2, p1, acc, n_erased);
  }
  return acc;
}

__device__ __forceinline__ void push_overflow(const ScoreParams& P, int r) {
  const uint32_t slot = atomicAdd(P.ovf_count, 1u);
  if (slot < P.ovf_cap) P.ovf_list[slot] = (uint32_t)r;
  else atomicOr(P.error_flag, 1u);
}

// FULL, tier 1 (the streaming kernel): every read of the shard is re-scored from an empty state and the total
// is reduced in the same pass (CalcScoreForPathsNew on a fresh ScoringState + GetTotalProb); the tile body is
// tier1_body below. Reads that own more than one record on a mate are a STATIC property of the cache: they are skipped
// there (idle lanes, no divergent code) and handled densely by tier 2 from a list built at commit time. A key that occurs
// several times in this evaluation (repeat node) leaves the read to paired_multi_kernel.

// FULL, tier 2 (second phase of the streaming kernel): the reads that own exactly two records on a mate and at most two on the other — (1,2), (2,1), (2,2)
// and the pairless (0,2), (2,0) — from a list built once per cache commit, class ordered, so a warp holds reads of ONE
// shape and the kernel is straight-line code with compile-time record counts. The records sit in a compact copy in
// list order; within a class every read owns the same number of rows, so the row addresses follow from the list index
// alone and the rows are requested together with the read's descriptor (three memory levels per read, like tier 1:
// {descriptor, rows} -> slot words -> pow/insert tables). Reads with three or more records on a mate are rare and go
// to paired_multi_kernel's static list.
struct Placed1 { bool live; bool multi; int walk, pos, edor; };
__device__ __forceinline__ Placed1 place_row(const ScoreParams& P, int m, const int4& rw) {
  Placed1 p;
  const int4 a = ldg4(P.m[m].slots_a + rw.x);   // {epoch | multi<<31, walk, cur_pos, skip_below}
  const uint32_t ef = (uint32_t)a.x;
  p.live = (ef & 0x7fffffffu) == P.epoch;
  p.multi = p.live && (ef >> 31);
  p.walk = a.y;
  p.pos = wrap_add(rw.y, a.z);
  if (p.pos < a.w) p.live = false;   // graph.cc:577
  p.edor = rw.z;
  return p;
}

// One tier-2 read with N1 / N2 records. 1 = scored (acc), 0 = belongs to paired_multi_kernel (a live key occurs
// several times), -1 = needs the enumeration order (many-placement pass).
// The state starts from 0 and every walk is "added" (full evaluation), so with at most two non-dropped pair terms the
// sum is order independent (0+a+b == 0+b+a). A duplicate placement (same walk, same position) with an identical
// payload is dropped whichever record is "later"; one with a different payload, or three and more terms, need the order.
template <int N1, int N2>
__device__ __forceinline__ int tier2_read(const ScoreParams& P, const RowShort* __restrict__ rows1,
                                          const RowShort* __restrict__ rows2, uint32_t b1, uint32_t b2, uint32_t ll, double& acc) {
  acc = 0.0;
  if (N1 == 0 || N2 == 0) return 1;   // no record on a mate: no pair term
  const int4 rx0 = ldg4(rows1 + b1), rx1 = N1 > 1 ? ldg4(rows1 + b1 + 1) : rx0;
  const int4 ry0 = ldg4(rows2 + b2), ry1 = N2 > 1 ? ldg4(rows2 + b2 + 1) : ry0;
  Placed1 x0 = place_row(P, 0, rx0), x1 = place_row(P, 0, rx1);
  Placed1 y0 = place_row(P, 1, ry0), y1 = place_row(P, 1, ry1);
  if (N1 < 2) x1.live = x1.multi = false;
  if (N2 < 2) y1.live = y1.multi = false;
  if (x0.multi || x1.multi || y0.multi || y1.multi) return 0;
  if (N1 > 1 && x0.live && x1.live && x0.walk == x1.walk && x0.pos == x1.pos) {
    if (x0.edor == x1.edor) x1.live = false; else return -1;
  }
  if (N2 > 1 && y0.live && y1.live && y0.walk == y1.walk && y0.pos == y1.pos) {
    if (y0.edor == y1.edor) y1.live = false; else return -1;
  }
  const int l1 = ll & 0xffff, l2 = ll >> 16;
  double t0 = 0.0, t1 = 0.0;   // the first two non-dropped terms
  int w0 = 0, xp0 = 0, yp0 = 0, w1 = 0, xp1 = 0, yp1 = 0;
  int nt = 0;
  const double px0 = align_prob(P.m[0], x0.edor, l1), px1 = N1 > 1 ? align_prob(P.m[0], x1.edor, l1) : 0.0;
  double tt;
#define GAML_TRY_PAIR(X, Y, PX)                                                                                         \
  if (X.live && Y.live && X.walk == Y.walk && pair_term(P, -1, X.pos, X.edor, Y.pos, Y.edor, l1, l2, PX, tt)) {         \
    if (nt == 0) { t0 = tt; w0 = X.walk; xp0 = X.pos; yp0 = Y.pos; }                                                    \
    else if (nt == 1) { t1 = tt; w1 = X.walk; xp1 = X.pos; yp1 = Y.pos; }                                               \
    nt++;                                                                                                               \
  }
  GAML_TRY_PAIR(x0, y0, px0)
  if (N2 > 1) { GAML_TRY_PAIR(x0, y1, px0) }
  if (N1 > 1) { GAML_TRY_PAIR(x1, y0, px1) }
  if (N1 > 1 && N2 > 1) { GAML_TRY_PAIR(x1, y1, px1) }
#undef GAML_TRY_PAIR
  if (nt > 2) return -1;
  if (nt >= 1) { acc = __dadd_rn(acc, t0); emit_cov(P, w0, xp0, yp0, l2, t0); }
  if (nt == 2) { acc = __dadd_rn(acc, t1); emit_cov(P, w1, xp1, yp1, l2, t1); }
  return 1;
}

// Tier-2 phase of the streaming kernel: tiles of 256 list entries, a block's first tile is its own index.
__device__ __forceinline__ void tier2_tiles(const ScoreParams& P, int* s_tile, Acc& sum, unsigned& floored) {
  const RowShort* rows1 = static_cast<const RowShort*>(P.m[0].crows);
  const RowShort* rows2 = static_cast<const RowShort*>(P.m[1].crows);
  const int n_tiles = (P.n_main + kBlock - 1) / kBlock;
  int tile = blockIdx.x, buf = 0;
  for (; tile < n_tiles; __syncthreads(), tile = s_tile[buf], buf ^= 1) {
    if (threadIdx.x == 0) s_tile[buf] = (int)gridDim.x + (int)atomicAdd(P.tile_counter + 2, 1u);
    const int k = tile * kBlock + (int)threadIdx.x;
    if (k >= P.n_main) continue;
    // list classes in order: (1,2) (2,1) (2,2) (0,2) (2,0); descriptor {read, packed lengths, -, -}
    int cls = 0;
#pragma unroll
    for (int c = 1; c < 5; c++) cls += (k >= P.class_begin[c]) ? 1 : 0;
    const uint32_t j = (uint32_t)(k - P.class_begin[cls]);
    const int4 dsc = ldg4(static_cast<const int4*>(P.cdesc) + k);
    const int r = dsc.x;
    const uint32_t ll = (uint32_t)dsc.y;
    double acc;
    int st;
    switch (cls) {
      case 0: st = tier2_read<1, 2>(P, rows1, rows2, P.cbase[0][0] + j, P.cbase[1][0] + 2 * j, ll, acc); break;
      case 1: st = tier2_read<2, 1>(P, rows1, rows2, P.cbase[0][1] + 2 * j, P.cbase[1][1] + j, ll, acc); break;
      case 2: st = tier2_read<2, 2>(P, rows1, rows2, P.cbase[0][2] + 2 * j, P.cbase[1][2] + 2 * j, ll, acc); break;
      default: st = 1; acc = 0.0; break;   // (0,2), (2,0): no pair term
    }
    if (P.dirty && __ldg(P.dirty + r)) continue;   // gained records since the list was built: the appendix phase's read
    if (st > 0) {
      P.values[r] = acc;
      acc_read(P, sum, floored, acc, (ll & 0xffff) + (ll >> 16));
    } else if (st < 0) {
      push_overflow(P, r);
    }
  }
}

// ---- tier 2 from packed entries ----------------------------------------------------------------------------------
// Packed copy of the tier-2 list's classes (1,2), (2,1), (2,2), built at commit when every record fits: a record is
// 8 bytes {key | edit<<22 | orient<<29, pos}; an entry is 2 (three records) or 3 (four records) uint4 units, stored unit
// major per class so that every unit load of a warp is one coalesced request:
//   (1,2): u0 = {read, lengths, x0}        u1 = {y0, y1}
//   (2,1): u0 = {read, lengths, y0}        u1 = {x0, x1}
//   (2,2): u0 = {read, lengths, -, -}      u1 = {x0, x1}      u2 = {y0, y1}
// 40 / 48 bytes per read instead of a 16-byte descriptor plus 48 / 64 bytes of rows.
struct Rec8 { uint32_t w; int pos; };
__device__ __forceinline__ Rec8 rec8(uint32_t a, uint32_t b) { return Rec8{a, (int)b}; }

// One tier-2 read, written like the tier-1 bodies: every load that does not depend on another is requested at once (slot
// words of all records; then, for all record combinations, the pair term and its logarithm from the set's term table —
// or the probability-table entries and the insert pdf when the set has none), filters are predicates, no branches.
// Same rules as tier2_read: status 1 = scored (acc), 0 = a live key occurs several times (the multi pass's read),
// -1 = the enumeration order matters (duplicate placement with a different payload, or three and more pair terms).
// qv = the fixed-point logarithm of acc when exactly one tabulated term makes up the value (else kTermOdd: take the log).
template <int N1, int N2>
__device__ __forceinline__ int tier2_packed_read(const ScoreParams& P, const int4* __restrict__ sa1, const int4* __restrict__ sa2,
                                                 const Rec8 (&x)[2], const Rec8 (&y)[2], uint32_t ll, double& acc, long long& qv) {
  const int l1 = ll & 0xffff, l2 = ll >> 16;
  int4 ox[2], oy[2];
#pragma unroll
  for (int i = 0; i < 2; i++) {
    ox[i] = __ldg(sa1 + (x[i < N1 ? i : 0].w & kPackKeyMask));
    oy[i] = __ldg(sa2 + (y[i < N2 ? i : 0].w & kPackKeyMask));
  }
  int ex[2], ey[2];
#pragma unroll
  for (int i = 0; i < 2; i++) {
    ex[i] = (int)((x[i < N1 ? i : 0].w >> kPackKeyBits) & kPackEdMask);
    ey[i] = (int)((y[i < N2 ? i : 0].w >> kPackKeyBits) & kPackEdMask);
  }
  const TermEntry* __restrict__ tq = P.tq ? static_cast<const TermEntry*>(P.tq) + 1 : nullptr;   // (entry 0: the fast records' "no pair term")
  double px[2], py[2];
  if (!tq) {
#pragma unroll
    for (int i = 0; i < 2; i++) {
      px[i] = __dmul_rn(__ldg(P.m[0].pow_mismatch + ex[i]), __ldg(P.m[0].pow_match + (l1 - ex[i])));
      py[i] = __dmul_rn(__ldg(P.m[1].pow_mismatch + ey[i]), __ldg(P.m[1].pow_match + (l2 - ey[i])));
    }
  }
  bool lx[2], ly[2], multi = false;
  int wx[2], wy[2], qx[2], qy[2], orx[2], ory[2];
#pragma unroll
  for (int i = 0; i < 2; i++) {
    const uint32_t fx = (uint32_t)ox[i].x, fy = (uint32_t)oy[i].x;
    const bool hx = i < N1, hy = i < N2;
    const bool vx = hx && (fx & 0x7fffffffu) == P.epoch, vy = hy && (fy & 0x7fffffffu) == P.epoch;
    multi |= (vx && (fx >> 31)) || (vy && (fy >> 31));
    wx[i] = ox[i].y; wy[i] = oy[i].y;
    qx[i] = wrap_add(x[hx ? i : 0].pos, ox[i].z); qy[i] = wrap_add(y[hy ? i : 0].pos, oy[i].z);
    lx[i] = vx && qx[i] >= ox[i].w;   // graph.cc:577
    ly[i] = vy && qy[i] >= oy[i].w;
    orx[i] = (int)((x[hx ? i : 0].w >> 29) & 1u); ory[i] = (int)((y[hy ? i : 0].w >> 29) & 1u);
  }
  bool order = false;
  if (N1 > 1) {   // duplicate placement: identical payload -> dropped, different payload -> the order decides
    const bool dup = lx[0] && lx[1] && wx[0] == wx[1] && qx[0] == qx[1];
    const bool same = ((x[0].w ^ x[1].w) >> kPackKeyBits) == 0u;
    order |= dup && !same;
    lx[1] = lx[1] && !dup;
  }
  if (N2 > 1) {
    const bool dup = ly[0] && ly[1] && wy[0] == wy[1] && qy[0] == qy[1];
    const bool same = ((y[0].w ^ y[1].w) >> kPackKeyBits) == 0u;
    order |= dup && !same;
    ly[1] = ly[1] && !dup;
  }
  bool ok[2][2];
  int dist[2][2];
  int nt = 0, nok = 0;
#pragma unroll
  for (int i = 0; i < N1; i++) {
#pragma unroll
    for (int j = 0; j < N2; j++) {
      const bool fwd = qx[i] < qy[j];
      const int d = fwd ? qy[j] - qx[i] + l2 : qx[i] - qy[j] + l1;   // graph.cc:1866-1875
      const bool term = lx[i] && ly[j] && wx[i] == wy[j] && orx[i] != ory[j] && orx[i] == (fwd ? 0 : 1);
      nt += term ? 1 : 0;
      ok[i][j] = term && (unsigned)d < (unsigned)P.ins_n;
      nok += ok[i][j] ? 1 : 0;
      dist[i][j] = ok[i][j] ? d : 0;
    }
  }
  double t[2][2];
  long long tqv[2][2];
  if (tq) {
    const int lim = 1 << P.tq_shift;
    bool untab = false;   // an edit distance beyond the table: (p1*p2)*ins from the probability tables instead
    TermEntry e[2][2];
#pragma unroll
    for (int i = 0; i < N1; i++) {
#pragma unroll
      for (int j = 0; j < N2; j++) {
        const bool fit = ex[i] < lim && ey[j] < lim;
        untab |= ok[i][j] && !fit;
        const size_t idx = fit ? (size_t)((ex[i] << P.tq_shift) | ey[j]) * (size_t)P.ins_n + (size_t)dist[i][j] : 0;
        const int4 w = __ldg(reinterpret_cast<const int4*>(tq + idx));
        e[i][j].t = __hiloint2double(w.y, w.x);
        e[i][j].q = (long long)(((unsigned long long)(uint32_t)w.w << 32) | (uint32_t)w.z);
      }
    }
#pragma unroll
    for (int i = 0; i < N1; i++) {
#pragma unroll
      for (int j = 0; j < N2; j++) { t[i][j] = e[i][j].t; tqv[i][j] = e[i][j].q; }
    }
    if (untab) {
#pragma unroll
      for (int i = 0; i < N1; i++) {
#pragma unroll
        for (int j = 0; j < N2; j++) {
          if (ok[i][j] && !(ex[i] < lim && ey[j] < lim)) {
            t[i][j] = __dmul_rn(__dmul_rn(__ldg(P.uni_prob[0] + ex[i]), __ldg(P.uni_prob[1] + ey[j])), __ldg(P.ins_tab + dist[i][j]));
            tqv[i][j] = kTermOdd;
          }
        }
      }
    }
  } else {
#pragma unroll
    for (int i = 0; i < N1; i++) {
#pragma unroll
      for (int j = 0; j < N2; j++) {
        t[i][j] = __dmul_rn(__dmul_rn(px[i], py[j]), __ldg(P.ins_tab + dist[i][j]));   // (p1*p2)*ins
        tqv[i][j] = kTermOdd;
      }
    }
  }
  // at most two terms survive below: 0 + a + b in any order is the same double, and absent terms are exact zeros
  acc = 0.0;
  qv = kTermOdd;
#pragma unroll
  for (int i = 0; i < N1; i++) {
#pragma unroll
    for (int j = 0; j < N2; j++) {
      acc = __dadd_rn(acc, ok[i][j] ? t[i][j] : 0.0);
      if (ok[i][j] && nok == 1) qv = tqv[i][j];
    }
  }
  return multi ? 0 : ((order || nt > 2) ? -1 : 1);
}

// Adds the term of a value whose fixed-point logarithm may be known already (qv != kTermOdd).
__device__ __forceinline__ void acc_term_known(Acc& a, unsigned& floored, const double2* log_tab, double p, long long qv,
                                               double pstar, long long qthr) {
  if (p < pstar) {
    floored++;
    acc_add_q(a, qthr);
  } else if (qv != kTermOdd) {
    acc_add_q(a, qv);
  } else {
    const double lg = table_log(log_tab, p);
    if (fabs(lg) < kFixLimit) acc_add_q(a, __double2ll_rn(lg * kFixScale));
    else acc_count_odd(a, lg);
  }
}

// Tier-2 phase from the packed entries: tiles of 256 list entries, a block's first tile is its own index.
__device__ __forceinline__ void tier2_packed_tiles(const ScoreParams& P, int* s_tile, Acc& sum, unsigned& floored) {
  const int4* sa1 = reinterpret_cast<const int4*>(P.m[0].slots_a);
  const int4* sa2 = reinterpret_cast<const int4*>(P.m[1].slots_a);
  const double2* log_tab = static_cast<const double2*>(P.log_tab);
  const uint4* __restrict__ pk = static_cast<const uint4*>(P.t2pack);
  const int n_tiles = (P.n_main + kBlock - 1) / kBlock;
  int tile = blockIdx.x, buf = 0;
  for (; tile < n_tiles; __syncthreads(), tile = s_tile[buf], buf ^= 1) {
    if (threadIdx.x == 0) s_tile[buf] = (int)gridDim.x + (int)atomicAdd(P.tile_counter + 2, 1u);
    const int k = tile * kBlock + (int)threadIdx.x;
    if (k >= P.n_main) continue;
    int cls = 0;
#pragma unroll
    for (int c = 1; c < 5; c++) cls += (k >= P.class_begin[c]) ? 1 : 0;
    const uint32_t j = (uint32_t)(k - P.class_begin[cls]);
    int r, st;
    uint32_t ll;
    double acc = 0.0;
    long long qv = kTermOdd;
    if (cls < 3) {
      const uint32_t n_c = (uint32_t)(P.class_begin[cls + 1] - P.class_begin[cls]);
      const uint4* base = pk + P.t2base[cls];
      const uint4 u0 = ldg_stream(base + j), u1 = ldg_stream(base + n_c + j);
      r = (int)u0.x;
      ll = u0.y;
      if (cls == 0) {
        const Rec8 x[2] = {rec8(u0.z, u0.w), rec8(u0.z, u0.w)}, y[2] = {rec8(u1.x, u1.y), rec8(u1.z, u1.w)};
        st = tier2_packed_read<1, 2>(P, sa1, sa2, x, y, ll, acc, qv);
      } else if (cls == 1) {
        const Rec8 x[2] = {rec8(u1.x, u1.y), rec8(u1.z, u1.w)}, y[2] = {rec8(u0.z, u0.w), rec8(u0.z, u0.w)};
        st = tier2_packed_read<2, 1>(P, sa1, sa2, x, y, ll, acc, qv);
      } else {
        const uint4 u2 = ldg_stream(base + 2 * n_c + j);
        const Rec8 x[2] = {rec8(u1.x, u1.y), rec8(u1.z, u1.w)}, y[2] = {rec8(u2.x, u2.y), rec8(u2.z, u2.w)};
        st = tier2_packed_read<2, 2>(P, sa1, sa2, x, y, ll, acc, qv);
      }
    } else {   // (0,2), (2,0): no pair term
      const int4 dsc = ldg4(static_cast<const int4*>(P.cdesc) + k);
      r = dsc.x;
      ll = (uint32_t)dsc.y;
      st = 1;
    }
    if (P.dirty && __ldg(P.dirty + r)) continue;   // gained records since the list was built: the appendix phase's read
    if (st > 0) {
      P.values[r] = acc;
      double pstar;
      long long qthr;
      term_consts(P, (ll & 0xffff) + (ll >> 16), pstar, qthr);
      acc_term_known(sum, floored, log_tab, acc, qv, pstar, qthr);
    } else if (st < 0) {
      push_overflow(P, r);
    }
  }
}

// Rare-shape phase of the streaming kernel: the listed reads with three or more records on a mate (list entries
// [n_main, n_complex)). Their records are walked in a loop — row from the compact copy, then its slot word — keeping
// at most two live, distinct placements per mate, which is what nearly all of them have in any one evaluation (most of
// a read's extra records sit under keys of joins that are not part of the current walks). Same rules as tier2_read:
// a live key that occurs several times -> the read is the multi pass's; anything that needs the enumeration order
// (three live placements, a duplicate with a different payload, three pair terms) -> many-placement pass.
struct TwoLive { Placed1 p0, p1; int n; bool multi, order; };
__device__ __forceinline__ void two_live_scan(const ScoreParams& P, int m, const RowShort* __restrict__ rows, uint32_t b,
                                              uint32_t n, TwoLive& t) {
  t.n = 0;
  t.multi = t.order = false;
  t.p0 = t.p1 = Placed1{false, false, 0, 0, 0};   // (pair_up indexes the pow tables with edor even for absent placements)
  for (uint32_t i = 0; i < n; i += 2) {   // two rows per step: their slot words are requested together
    const int4 r0 = ldg4(rows + b + i), r1 = i + 1 < n ? ldg4(rows + b + i + 1) : r0;
    Placed1 q[2] = {place_row(P, m, r0), place_row(P, m, r1)};
    if (i + 1 >= n) q[1].live = q[1].multi = false;
#pragma unroll
    for (int j = 0; j < 2; j++) {
      if (!q[j].live) continue;
      t.multi |= q[j].multi;
      if (t.n > 0 && t.p0.walk == q[j].walk && t.p0.pos == q[j].pos) {
        if (t.p0.edor != q[j].edor) t.order = true;
      } else if (t.n > 1 && t.p1.walk == q[j].walk && t.p1.pos == q[j].pos) {
        if (t.p1.edor != q[j].edor) t.order = true;
      } else if (t.n == 0) {
        t.p0 = q[j];
        t.n = 1;
      } else if (t.n == 1) {
        t.p1 = q[j];
        t.n = 2;
      } else {
        t.order = true;
      }
    }
  }
}

// Pair terms of up to two live placements per mate; false when three or more terms survive (order matters then).
__device__ __forceinline__ bool pair_up(const ScoreParams& P, const Placed1& x0, const Placed1& x1, const Placed1& y0,
                                        const Placed1& y1, uint32_t ll, double& acc) {
  const int l1 = ll & 0xffff, l2 = ll >> 16;
  double t0 = 0.0, t1 = 0.0;   // the first two non-dropped terms
  int w0 = 0, xp0 = 0, yp0 = 0, w1 = 0, xp1 = 0, yp1 = 0;
  int nt = 0;
  const double px0 = align_prob(P.m[0], x0.edor, l1), px1 = align_prob(P.m[0], x1.edor, l1);
  double tt;
#define GAML_TRY_PAIR(X, Y, PX)                                                                                         \
  if (X.live && Y.live && X.walk == Y.walk && pair_term(P, -1, X.pos, X.edor, Y.pos, Y.edor, l1, l2, PX, tt)) {         \
    if (nt == 0) { t0 = tt; w0 = X.walk; xp0 = X.pos; yp0 = Y.pos; }                                                    \
    else if (nt == 1) { t1 = tt; w1 = X.walk; xp1 = X.pos; yp1 = Y.pos; }                                               \
    nt++;                                                                                                               \
  }
  GAML_TRY_PAIR(x0, y0, px0)
  GAML_TRY_PAIR(x0, y1, px0)
  GAML_TRY_PAIR(x1, y0, px1)
  GAML_TRY_PAIR(x1, y1, px1)
#undef GAML_TRY_PAIR
  if (nt > 2) return false;
  acc = 0.0;
  if (nt >= 1) { acc = __dadd_rn(acc, t0); emit_cov(P, w0, xp0, yp0, l2, t0); }
  if (nt == 2) { acc = __dadd_rn(acc, t1); emit_cov(P, w1, xp1, yp1, l2, t1); }
  return true;
}

__device__ __forceinline__ void rare_tiles(const ScoreParams& P, int* s_tile, Acc& sum, unsigned& floored) {
  const RowShort* rows1 = static_cast<const RowShort*>(P.m[0].crows);
  const RowShort* rows2 = static_cast<const RowShort*>(P.m[1].crows);
  const int n_rare = P.n_complex - P.n_main;
  const int n_tiles = (n_rare + kBlock - 1) / kBlock;
  int tile = blockIdx.x, buf = 0;
  for (; tile < n_tiles; __syncthreads(), tile = s_tile[buf], buf ^= 1) {
    if (threadIdx.x == 0) s_tile[buf] = (int)gridDim.x + (int)atomicAdd(P.tile_counter + 1, 1u);
    const int k = P.n_main + tile * kBlock + (int)threadIdx.x;
    if (k >= P.n_complex) continue;
    const int4 dsc = ldg4(static_cast<const int4*>(P.cdesc) + k);   // {read, packed lengths, first compact row mate 1, mate 2}
    const uint32_t e1 = __ldg(P.m[0].cptr + k + 1), e2 = __ldg(P.m[1].cptr + k + 1);
    const int r = dsc.x;
    const uint32_t ll = (uint32_t)dsc.y;
    if (P.dirty && __ldg(P.dirty + r)) continue;   // gained records since the list was built: the appendix phase's read
    TwoLive x, y;
    two_live_scan(P, 0, rows1, (uint32_t)dsc.z, e1 - (uint32_t)dsc.z, x);
    two_live_scan(P, 1, rows2, (uint32_t)dsc.w, e2 - (uint32_t)dsc.w, y);
    if (x.multi || y.multi) continue;   // the multi pass's read
    double acc = 0.0;
    if (x.order || y.order || !pair_up(P, x.p0, x.p1, y.p0, y.p1, ll, acc)) {
      push_overflow(P, r);
      continue;
    }
    P.values[r] = acc;
    acc_read(P, sum, floored, acc, (ll & 0xffff) + (ll >> 16));
  }
}

// Tier-1 tile body: kR reads per lane of one warp tile, every step written without branches so that the kR
// dependent chains (packed record -> {slot words, term-table entry} -> select -> accumulate) are issued side by side: one
// trip per memory level for all of them. The filters of the pair term (liveness, skip rule graph.cc:577, one walk,
// orientation/order graph.cc:1864-1875, insert-table range) are predicates (a dropped pair is a term of +0.0, which is
// what the state holds for such a read); the rare fix-ups (mates under different keys, an edit distance beyond the term
// table, a non-finite logarithm) are taken once, after the common work of all kR reads.
//   kTab: the set has a term table (uniform lengths) and a combined slot table: the pair term AND its fixed-point
//         logarithm come from ONE 16-byte gather, requested together with the slot words (for mates under the same key
//         the insert distance is a property of the two records: both share the key's offset in the walk);
//   else: the term is formed from the probability tables and the insert pdf, the logarithm by table_log.
template <bool kCov, bool kPacked, bool kTab, int kR>
__device__ __forceinline__ void tier1_body(const ScoreParams& P, const uint4* __restrict__ src1, const uint4* __restrict__ src2,
                                           int lane, const int4* __restrict__ sa1, const int4* __restrict__ sa2,
                                           const double2* __restrict__ log_tab, int q_first, int n, Acc& sum, unsigned& floored,
                                           const uint32_t* __restrict__ ridx = nullptr) {
  static_assert(!kTab || (kPacked && !kCov), "the term table goes with the packed pairs");
  // level 1: the records of this lane's kR reads (read q_first + 32 j + lane — or, with a list, the reads at those list
  // positions; positions past the end are clamped to the last one and masked out below) and the lengths unless the whole
  // set shares them
  int qi[kR];
  bool valid[kR];
#pragma unroll
  for (int j = 0; j < kR; j++) {
    const int q = q_first + 32 * j + lane;
    valid[j] = q < n;
    qi[j] = min(q, n - 1);
  }
  if (ridx) {
#pragma unroll
    for (int j = 0; j < kR; j++) qi[j] = (int)__ldg(ridx + qi[j]);
    if (P.dirty) {   // (a dirty read's packed pair carries the "elsewhere" flag: masked out below like a tier-2 read)
    }
  }
  uint4 u1[kR], u2[kR];
#pragma unroll
  for (int j = 0; j < kR; j++) {
    u1[j] = ldg_stream(src1 + qi[j]);
    if (!kPacked) u2[j] = ldg_stream(src2 + qi[j]);
  }
  int key1[kR], key2[kR], pos1[kR], pos2[kR], e1[kR], e2[kR], xo[kR], yo[kR];
  bool has1[kR], has2[kR], tier2[kR], same[kR];
  uint32_t ll[kR];
  if (kTab || P.lens_uniform) {
#pragma unroll
    for (int j = 0; j < kR; j++) ll[j] = P.uniform_ll;
  } else {
#pragma unroll
    for (int j = 0; j < kR; j++) ll[j] = __ldg(P.lens + qi[j]);
  }
  if (kPacked) {
#pragma unroll
    for (int j = 0; j < kR; j++) {
      const uint4 pr = u1[j];
      key1[j] = (int)(pr.x & kPackKeyMask);
      key2[j] = (int)(pr.y & kPackKeyMask);
      e1[j] = (int)((pr.x >> kPackKeyBits) & kPackEdMask);
      e2[j] = (int)((pr.y >> kPackKeyBits) & kPackEdMask);
      xo[j] = (int)((pr.x >> 29) & 1u);
      yo[j] = (int)((pr.y >> 29) & 1u);
      has1[j] = ((pr.x >> 30) & 1u) == 0u;
      has2[j] = ((pr.y >> 30) & 1u) == 0u;
      tier2[j] = (pr.x >> 31) != 0u;
      same[j] = (pr.y >> 31) != 0u;
      pos1[j] = (int)pr.z;
      pos2[j] = (int)pr.w;
    }
  } else {
#pragma unroll
    for (int j = 0; j < kR; j++) {
      const int4 rw1 = make_int4((int)u1[j].x, (int)u1[j].y, (int)u1[j].z, (int)u1[j].w);
      const int4 rw2 = make_int4((int)u2[j].x, (int)u2[j].y, (int)u2[j].z, (int)u2[j].w);
      key1[j] = max(rw1.x, 0);   // key -1 (no record) reads slot 0, ignored below
      key2[j] = max(rw2.x, 0);
      has1[j] = rw1.x >= 0;
      has2[j] = rw2.x >= 0;
      e1[j] = rw1.z & 0xffff;
      e2[j] = rw2.z & 0xffff;
      xo[j] = (rw1.z >> 30) & 1;
      yo[j] = (rw2.z >> 30) & 1;
      tier2[j] = (((rw1.z | rw2.z) >> 17) & 0x1fff) != 0;   // count >= 2 on a mate
      same[j] = false;
      pos1[j] = rw1.y;
      pos2[j] = rw2.y;
    }
  }
  // level 2: slot words of both keys (L1/L2 resident) and, with a term table, the entry the records themselves point at
  int4 o1[kR], o2[kR];
  if (kPacked && P.comb) {
    // one 256-bit gather per read: {mate 1's slot word, the same key's word in mate 2's store}; the few pairs whose mates
    // lie under different keys take mate 2's word from its own table (predicated second gather)
    const uint4* __restrict__ comb = static_cast<const uint4*>(P.comb);
#pragma unroll
    for (int j = 0; j < kR; j++) {
      uint4 a, b;
      ldg256(comb + 4 * key1[j], a, b);
      o1[j] = make_int4((int)a.x, (int)a.y, (int)a.z, (int)a.w);
      o2[j] = make_int4((int)b.x, (int)b.y, (int)b.z, (int)b.w);
    }
  } else {
#pragma unroll
    for (int j = 0; j < kR; j++) {
      o1[j] = __ldg(sa1 + key1[j]);
      o2[j] = __ldg(sa2 + key2[j]);
    }
  }
  const int4* __restrict__ tq = static_cast<const int4*>(P.tq) + 1;   // (entry 0 is the fast records' "no pair term")
  int4 te[kR];
  unsigned tix[kR];
  bool fit[kR];
  if (kTab) {
    const int lim = 1 << P.tq_shift;
#pragma unroll
    for (int j = 0; j < kR; j++) {
      const int l1 = ll[j] & 0xffff, l2 = ll[j] >> 16;
      const bool fwd = pos1[j] < pos2[j];
      const int d = fwd ? pos2[j] - pos1[j] + l2 : pos1[j] - pos2[j] + l1;
      fit[j] = e1[j] < lim && e2[j] < lim;
      tix[j] = (fit[j] && (unsigned)d < (unsigned)P.ins_n) ? (unsigned)((e1[j] << P.tq_shift) | e2[j]) * (unsigned)P.ins_n + (unsigned)d : 0u;
      te[j] = __ldg(tq + tix[j]);
    }
  }
  if (kPacked && P.comb) {
#pragma unroll
    for (int j = 0; j < kR; j++)
      if (!same[j]) o2[j] = __ldg(sa2 + key2[j]);
  }
  bool mine[kR], ok[kR];
  int dist[kR], px[kR], py[kR];
#pragma unroll
  for (int j = 0; j < kR; j++) {
    const int l1 = ll[j] & 0xffff, l2 = ll[j] >> 16;
    const uint32_t f1 = (uint32_t)o1[j].x, f2 = (uint32_t)o2[j].x;
    const bool live1 = has1[j] && (f1 & 0x7fffffffu) == P.epoch, live2 = has2[j] && (f2 & 0x7fffffffu) == P.epoch;
    const bool multi = (live1 && (f1 >> 31)) || (live2 && (f2 >> 31));             // paired_multi_kernel's read
    mine[j] = valid[j] && !tier2[j] && !multi;
    const int p1 = wrap_add(pos1[j], o1[j].z), p2 = wrap_add(pos2[j], o2[j].z);
    px[j] = p1;
    py[j] = p2;
    const bool fwd = p1 < p2;
    const int d = fwd ? p2 - p1 + l2 : p1 - p2 + l1;                               // graph.cc:1866-1875
    const bool placed = live1 && live2 && p1 >= o1[j].w && p2 >= o2[j].w && o1[j].y == o2[j].y;   // graph.cc:577; one walk
    ok[j] = mine[j] && placed && xo[j] != yo[j] && xo[j] == (fwd ? 0 : 1) && (unsigned)d < (unsigned)P.ins_n;
    dist[j] = ok[j] ? d : 0;
  }
  // floor test and floored term of each read (a kernel parameter when the whole set shares the lengths)
  double pstar[kR];
  long long qthr[kR];
#pragma unroll
  for (int j = 0; j < kR; j++) {
    if (kTab || P.lens_uniform) {
      pstar[j] = P.uni_pstar;
      qthr[j] = P.uni_qthr;
    } else {
      term_consts(P, (ll[j] & 0xffff) + (ll[j] >> 16), pstar[j], qthr[j]);
    }
  }
  // the pair term (p1*p2)*ins (graph.cc:1889) and, where known, its fixed-point logarithm
  double acc[kR];
  long long qv[kR];
  if (kTab) {
    bool again = false, untab = false;
#pragma unroll
    for (int j = 0; j < kR; j++) {
      const unsigned want = (unsigned)((e1[j] << P.tq_shift) | e2[j]) * (unsigned)P.ins_n + (unsigned)dist[j];
      again |= ok[j] && fit[j] && want != tix[j];   // mates under different keys: the distance depends on the walk
      untab |= ok[j] && !fit[j];
    }
    if (again) {
#pragma unroll
      for (int j = 0; j < kR; j++) {
        const unsigned want = (unsigned)((e1[j] << P.tq_shift) | e2[j]) * (unsigned)P.ins_n + (unsigned)dist[j];
        if (ok[j] && fit[j] && want != tix[j]) te[j] = __ldg(tq + want);
      }
    }
#pragma unroll
    for (int j = 0; j < kR; j++) {
      acc[j] = ok[j] ? __hiloint2double(te[j].y, te[j].x) : 0.0;
      qv[j] = (long long)(((unsigned long long)(uint32_t)te[j].w << 32) | (uint32_t)te[j].z);
    }
    if (untab) {
#pragma unroll
      for (int j = 0; j < kR; j++) {
        if (ok[j] && !fit[j]) {
          acc[j] = __dmul_rn(__dmul_rn(__ldg(P.uni_prob[0] + e1[j]), __ldg(P.uni_prob[1] + e2[j])), __ldg(P.ins_tab + dist[j]));
          qv[j] = fix_log(log_tab, acc[j]);
        }
      }
    }
  } else {
    double pa[kR], pb[kR];
    if (kPacked && P.uni_prob[0]) {
      // set-uniform lengths: the alignment probability depends on the edit distance alone (one table entry per mate)
#pragma unroll
      for (int j = 0; j < kR; j++) {
        pa[j] = __ldg(P.uni_prob[0] + e1[j]);
        pb[j] = __ldg(P.uni_prob[1] + e2[j]);
      }
    } else {
#pragma unroll
      for (int j = 0; j < kR; j++) {
        const int l1 = ll[j] & 0xffff, l2 = ll[j] >> 16;
        pa[j] = __dmul_rn(__ldg(P.m[0].pow_mismatch + e1[j]), __ldg(P.m[0].pow_match + (l1 - e1[j])));
        pb[j] = __dmul_rn(__ldg(P.m[1].pow_mismatch + e2[j]), __ldg(P.m[1].pow_match + (l2 - e2[j])));
      }
    }
#pragma unroll
    for (int j = 0; j < kR; j++) {
      const double ins = __ldg(P.ins_tab + dist[j]);
      const double t = __dmul_rn(__dmul_rn(pa[j], pb[j]), ins);                        // (p1*p2)*ins, graph.cc:1889
      acc[j] = ok[j] ? t : 0.0;                                                        // a full evaluation only adds: 0 + t
      if (kCov) {
        if (ok[j]) emit_cov(P, o1[j].y, px[j], py[j], (int)(ll[j] >> 16), t);
      }
    }
    // table_log's fast path, computed unconditionally (garbage, not a trap, for 0/denormal/non-finite input)
    bool special = false;
    double lg[kR];
#pragma unroll
    for (int j = 0; j < kR; j++) {
      const long long ix = __double_as_longlong(acc[j]);
      special |= mine[j] && !(acc[j] < pstar[j]) && (unsigned long long)(ix - 0x0010000000000000ll) >= 0x7fe0000000000000ull;
      const long long tmp = ix - 0x3fe6000000000000ll;
      const int i = (int)((tmp >> 45) & 127);
      const long long k = tmp >> 52;
      const double z = __longlong_as_double(ix - (tmp & 0xfff0000000000000ll));
      const double2 e = log_tab[i];
      const double r = fma(z, e.x, -1.0);
      double p = fma(r, 1.0 / 7.0, -1.0 / 6.0);
      p = fma(r, p, 0.2);
      p = fma(r, p, -0.25);
      p = fma(r, p, 1.0 / 3.0);
      p = fma(r, p, -0.5);
      p = fma(r * r, p, r);
      lg[j] = fma((double)k, 0.693147180559945309417232121458, e.y) + p;
    }
    if (special) {
#pragma unroll
      for (int j = 0; j < kR; j++) {
        const long long ix = __double_as_longlong(acc[j]);
        if (!(acc[j] < pstar[j]) && (unsigned long long)(ix - 0x0010000000000000ll) >= 0x7fe0000000000000ull) lg[j] = slow_log(acc[j]);
      }
    }
#pragma unroll
    for (int j = 0; j < kR; j++) qv[j] = fabs(lg[j]) < kFixLimit ? __double2ll_rn(lg[j] * kFixScale) : kTermOdd;
  }
  // floor test, state write, exact accumulation
  bool odd = false;   // a term outside the fixed-point range (log 0 = -inf, NaN): counted, not added
#pragma unroll
  for (int j = 0; j < kR; j++) {
    if (mine[j]) P.values[qi[j]] = acc[j];
    const bool fl = acc[j] < pstar[j];
    const long long q = fl ? qthr[j] : qv[j];
    const bool fin = q != kTermOdd;
    odd |= mine[j] && !fin;
    acc_add_q(sum, (mine[j] && fin) ? q : 0ll);
    floored += (mine[j] && fl) ? 1u : 0u;
  }
  if (odd) {
#pragma unroll
    for (int j = 0; j < kR; j++)
      if (mine[j] && !(acc[j] < pstar[j]) && qv[j] == kTermOdd) acc_count_odd(sum, table_log(log_tab, acc[j]));
  }
}

// Tier-1 tile body over FastPair records (sets with a term table): per read one 16-byte record, one 32-byte gather of the
// key's two slot words and one 16-byte gather of the term-table entry the record points at — both gathers depend on the
// record only, so a tile is two memory levels — then liveness and the skip rule (graph.cc:577) as predicates, the select,
// the state write and the exact accumulation. Everything else about the pair was resolved when the cache was committed.
template <int kR>
__device__ __forceinline__ void tier1_fast_load(const uint4* __restrict__ fast, int lane, int q_first, int n, uint4 (&u)[kR]) {
#pragma unroll
  for (int j = 0; j < kR; j++) u[j] = ldg_stream(fast + min(q_first + 32 * j + lane, n - 1));
}
template <int kR>
__device__ __forceinline__ void tier1_fast(const ScoreParams& P, const uint4 (&u)[kR], int lane, int q_first, int n, Acc& sum,
                                           unsigned& floored, const double2* __restrict__ log_tab) {
  int qi[kR];
  bool valid[kR];
#pragma unroll
  for (int j = 0; j < kR; j++) {
    const int q = q_first + 32 * j + lane;
    valid[j] = q < n;
    qi[j] = min(q, n - 1);
  }
  const uint4* __restrict__ comb = static_cast<const uint4*>(P.comb);
  const int4* __restrict__ tq = static_cast<const int4*>(P.tq);
  uint4 a[kR], b[kR];
  int4 te[kR];
#pragma unroll
  for (int j = 0; j < kR; j++) {
    ldg256(comb + 4 * (u[j].x & 0x3fffffffu), a[j], b[j]);   // {epoch | multi << 31, walk, cur_pos, skip_below} of both mates
    te[j] = __ldg(tq + u[j].w);
  }
  const double pstar = P.uni_pstar;
  const long long qthr = P.uni_qthr;
  bool odd = false;
  double val[kR];
  long long qv[kR];
  bool mine[kR];
#pragma unroll
  for (int j = 0; j < kR; j++) {
    const bool elsewhere = (u[j].x >> 31) != 0u, noterm = ((u[j].x >> 30) & 1u) != 0u;
    const bool live = !noterm && (a[j].x & 0x7fffffffu) == P.epoch && (b[j].x & 0x7fffffffu) == P.epoch;
    const bool multi = live && (((a[j].x | b[j].x) >> 31) != 0u);                       // paired_multi_kernel's read
    mine[j] = valid[j] && !elsewhere && !multi;
    const bool ok = live && wrap_add((int)u[j].y, (int)a[j].z) >= (int)a[j].w && wrap_add((int)u[j].z, (int)b[j].z) >= (int)b[j].w &&
                    a[j].y == b[j].y;                                                   // graph.cc:577; one walk
    val[j] = ok ? __hiloint2double(te[j].y, te[j].x) : 0.0;
    qv[j] = (long long)(((unsigned long long)(uint32_t)te[j].w << 32) | (uint32_t)te[j].z);
  }
#pragma unroll
  for (int j = 0; j < kR; j++) {
    if (mine[j]) P.values[qi[j]] = val[j];
    const bool fl = val[j] < pstar;
    const long long q = fl ? qthr : qv[j];
    const bool fin = q != kTermOdd;
    odd |= mine[j] && !fin;
    acc_add_q(sum, (mine[j] && fin) ? q : 0ll);
    floored += (mine[j] && fl) ? 1u : 0u;
  }
  if (odd) {   // a value whose logarithm is not finite (0 under a zero threshold): counted, not added
#pragma unroll
    for (int j = 0; j < kR; j++)
      if (mine[j] && !(val[j] < pstar) && qv[j] == kTermOdd) acc_count_odd(sum, table_log(log_tab, val[j]));
  }
}

// FULL, the streaming kernel: tier 1 (every read with at most one record per mate, straight from the dense
// first-record arrays) and then tier 2 (the static list of reads with two records on a mate, from the compact copy) in
// one launch — both are tile loops over static data drawn from counters, so a block simply moves on to tier-2 tiles when
// the tier-1 tiles run out, without a kernel boundary (ramp, tail, launch) in between.
// kPhase: 0 = every phase in one launch; sets with fast records run TWO launches back to back in the chain — 1 = tier 1
// over the fast records alone (a light body: twice the resident warps of the fused kernel, and tier 1 is bound by memory
// latency), 2 = everything else (rare shapes, cross list, tier 2, appendix).
template <bool kCov, bool kPacked, bool kTab, int kBPS, int kR, int kPhase = 0>
__global__ void __launch_bounds__(kBlock, kBPS) paired_stream_kernel(const ScoreParams P) {
  tl_begin(P.timeline, kPhase == 2 ? kTlTier2 : kTlTier1);
  const int4* sa1 = reinterpret_cast<const int4*>(P.m[0].slots_a);
  const int4* sa2 = reinterpret_cast<const int4*>(P.m[1].slots_a);
  const double2* log_tab = static_cast<const double2*>(P.log_tab);
  Acc sum = acc_zero();
  unsigned floored = 0;
  const int n = P.n_reads;
  __shared__ int s_tile[2];
  // Tier 1: work is handed out in tiles of kR x 256 consecutive reads (a warp takes kR x 32 consecutive ones of them). A
  // block's first two tiles are static (its own index, then + gridDim), the rest is drawn from a counter (zeroed by
  // apply_slots) TWO tiles ahead: blocks that become resident late — the multi pass in front of this kernel holds part of
  // the register file for a while — or run slowly simply take fewer tiles, and the next tile's lines are pulled into L2
  // (prefetch.global.L2, no registers held) while the current tile is being worked on, so its demand loads find them
  // there. The exact integer accumulators make the result independent of who sums what.
  constexpr int kTile = kR * kBlock;
  constexpr int kRecLines = kTile * 16 / 128;   // 128-byte lines of one record array per tile
  const int n1 = kTab ? P.n_tier1 : n;          // fast records: tier 1 ends with the last fast read of the internal order
  const int n_tiles = (n1 + kTile - 1) / kTile;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const uint4* __restrict__ src1 = static_cast<const uint4*>(kTab ? P.fast : (kPacked ? P.pairs : P.m[0].first));
  const uint4* __restrict__ src2 = static_cast<const uint4*>(P.m[1].first);
  auto prefetch_tile = [&](int t) {
    if (t >= n_tiles) return;
    const int q = min(t * kTile + ((int)threadIdx.x % kRecLines) * 8, n1 - 1);   // 8 consecutive 16-byte records = one line
    if ((int)threadIdx.x < kRecLines) prefetch_l2(src1 + q);
    else if (!kPacked && (int)threadIdx.x < 2 * kRecLines) prefetch_l2(src2 + q);
  };
  static_assert(2 * kRecLines <= kBlock, "one prefetch per thread");
  int tile = blockIdx.x, next = (int)blockIdx.x + (int)gridDim.x, buf = 0;
  if (kPhase != 2) prefetch_tile(tile);   // static data: may be requested before the wait below
  // First kernel after apply_slots (no multi pass before it): wait here, release after. Otherwise the multi pass did
  // that, every block of this kernel starts after apply_slots completed, and the wait moves to the end.
  if (P.chain_first) pdl_wait();
  pdl_release();   // AFTER the wait: the next streaming kernel starts without a wait of its own, see tier 2
  // The rare-shape tiles go first: their long dependent chains overlap with everything after them instead of forming
  // the kernel's tail.
  if (kPhase != 1 && P.n_complex > P.n_main) {
    rare_tiles(P, s_tile, sum, floored);
    __syncthreads();
  }
  if (kPhase == 2) {
    // (tier 1 runs in the launch before this one)
  } else if (kTab) {
    // fast records: the NEXT tile's records are requested into registers before this tile is worked on (a tile is two
    // memory levels: its records, then the gathers they point at — the first level is always one tile ahead)
    uint4 u_cur[kR], u_nxt[kR];
    if (tile < n_tiles) tier1_fast_load<kR>(src1, lane, tile * kTile + wib * (32 * kR), n1, u_cur);
    while (tile < n_tiles) {
      if (threadIdx.x == 0) s_tile[buf] = 2 * (int)gridDim.x + (int)atomicAdd(P.tile_counter, 1u);   // the tile after next
      if (next < n_tiles) tier1_fast_load<kR>(src1, lane, next * kTile + wib * (32 * kR), n1, u_nxt);
      tier1_fast<kR>(P, u_cur, lane, tile * kTile + wib * (32 * kR), n1, sum, floored, log_tab);
      __syncthreads();
#pragma unroll
      for (int j = 0; j < kR; j++) u_cur[j] = u_nxt[j];
      tile = next;
      next = s_tile[buf];
      buf ^= 1;
    }
  } else {
    while (tile < n_tiles) {
      if (threadIdx.x == 0) s_tile[buf] = 2 * (int)gridDim.x + (int)atomicAdd(P.tile_counter, 1u);   // the tile after next
      prefetch_tile(next);
      tier1_body<kCov, kPacked, false, kR>(P, src1, src2, lane, sa1, sa2, log_tab, tile * kTile + wib * (32 * kR), n, sum, floored);
      __syncthreads();
      tile = next;
      next = s_tile[buf];
      buf ^= 1;
    }
  }
  if (kPhase != 1 && kTab && P.n_cross > 0) {
    // the cross list: tier-1 reads whose mates lie under different keys (the insert distance depends on the walk) or whose
    // edit distance is beyond the term table — the general body over the packed pairs, read ids from the list
    const uint4* __restrict__ pairs = static_cast<const uint4*>(P.pairs);
    constexpr int kXR = 2, kXTile = kXR * kBlock;   // (two reads per lane whatever the fast tiles use: this body is the wide one)
    const int x_tiles = (P.n_cross + kXTile - 1) / kXTile;
    __syncthreads();
    int xt = blockIdx.x, xbuf = 0;
    for (; xt < x_tiles; __syncthreads(), xt = s_tile[xbuf], xbuf ^= 1) {
      if (threadIdx.x == 0) s_tile[xbuf] = (int)gridDim.x + (int)atomicAdd(P.tile_counter + 3, 1u);
      tier1_body<false, true, kTab, kXR>(P, pairs, src2, lane, sa1, sa2, log_tab, xt * kXTile + wib * (32 * kXR), P.n_cross, sum, floored, P.xlist);
    }
  }
  if (kPhase != 2) tl_end(P.timeline, kTlTier1);
  if (kPhase != 1 && P.n_main > 0) {
    __syncthreads();   // s_tile is shared with the rare-shape phase
    if (kPhase == 0) tl_begin(P.timeline, kTlTier2);
    if (!kCov && P.t2pack) tier2_packed_tiles(P, s_tile, sum, floored);
    else tier2_tiles(P, s_tile, sum, floored);
  }
  if (kPhase != 1) tl_end(P.timeline, kTlTier2);
  if (!P.chain_first) pdl_wait();
  block_accumulate(sum, floored, P.accum);
  if (P.finish_here) finish_set_if_complete(P);
}


// General replay of one read: the ordered register paths, then the scratch path (exact counts, scratch from a bump
// allocator). Returns false when the scratch arena is exhausted (error flag set).
__device__ __forceinline__ bool paired_read_any(const ScoreParams& P, int r, uint32_t ll, double& acc) {
  if (paired_read_ordered(P, r, acc)) return true;   // at most four LIVE placements per mate
  const int n1 = gather_short(P.m[0], P.epoch, r, nullptr), n2 = gather_short(P.m[1], P.epoch, r, nullptr);
  const unsigned long long base = atomicAdd(P.scratch_cursor, (unsigned long long)(n1 + n2));
  if (base + n1 + n2 > P.scratch_cap) {
    atomicOr(P.error_flag, 2u);
    return false;
  }
  Plc* a = P.scratch + base;
  Plc* b = a + n1;
  gather_short(P.m[0], P.epoch, r, a);
  gather_short(P.m[1], P.epoch, r, b);
  acc = apply_pairs(P, a, n1, b, n2, ll & 0xffff, ll >> 16, acc, P.n_erased);
  return true;
}

// FULL, multi pass: the reads a full evaluation cannot stream — every read with a record under a key that occurs
// several times in this evaluation (repeat nodes), enumerated from those keys' ranges of the key-major arenas of both
// mates, like the delta kernel does. A read reachable twice is claimed once through its stamp. It depends on apply_slots only, so it is the FIRST kernel
// of the chain after it: a small grid whose latency-bound, divergent work runs underneath the streaming kernels
// instead of after them.
__global__ void __launch_bounds__(kOvfBlock) paired_multi_kernel(const ScoreParams P) {
  tl_begin(P.timeline, kTlDelta);
  if (P.chain_first) pdl_wait();
  pdl_release();
  Acc sum = acc_zero();
  unsigned floored = 0;
  const uint32_t total = P.n_mtouch > 0 ? __ldg(P.mtouch_prefix + P.n_mtouch) : 0u;
  for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < total; q += gridDim.x * blockDim.x) {
    int lo = 0, hi = P.n_mtouch;   // largest t with prefix[t] <= q
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (__ldg(P.mtouch_prefix + mid) <= q) lo = mid; else hi = mid;
    }
    const TouchRange tr = P.mtouch[lo];
    const ArenaShort* arena = lo < P.n_mtouch1 ? P.arena1 : P.arena2;
    const int r = ldg4(arena + tr.begin + (q - __ldg(P.mtouch_prefix + lo))).x;
    if (atomicExch(P.stamp + r, P.epoch) == P.epoch) continue;   // reachable through several keys / both mates
    const uint32_t ll = __ldg(P.lens + r);
    double acc = 0.0;
    if (!paired_read_any(P, r, ll, acc)) continue;
    P.values[r] = acc;
    acc_read(P, sum, floored, acc, (ll & 0xffff) + (ll >> 16));
  }
  // the appendix: reads that gained records since the static lists were built (cache appends), scored from their
  // (relocated) rows by the same general path; one under a repeated key may have been claimed by the loop above
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < P.n_appx; k += gridDim.x * blockDim.x) {
    const int r = (int)__ldg(P.appx_list + k);
    if (atomicExch(P.stamp + r, P.epoch) == P.epoch) continue;
    const uint32_t ll = __ldg(P.lens + r);
    double acc = 0.0;
    if (!paired_read_any(P, r, ll, acc)) continue;
    P.values[r] = acc;
    acc_read(P, sum, floored, acc, (ll & 0xffff) + (ll >> 16));
  }
  if (!P.chain_first) pdl_wait();
  block_accumulate(sum, floored, P.accum);
  if (P.finish_here) finish_set_if_complete(P);
  tl_end(P.timeline, kTlDelta);
}

// Replay of a touched FAST read (one record per mate, both under one key, term resolved at commit — FastPair): its pair
// term T is a property of the two records, so the subtract/add sequence of graph.cc:1936-1950 is "T leaves for every
// erased walk that holds the key and passes the skip rule, T enters for every added one", in enumeration order. Everything
// comes from the 64-byte combined slot entry of the key (both words of both mates), at most one further occurrence per
// mate and the term-table entry: three memory levels instead of the general path's six. Covers keys that occur at most
// twice in the evaluation, in different walks (the normal case: once in the erased walk, once in the added one).
// Returns false when the general path has to take the read.
__device__ __forceinline__ bool delta_fast(const ScoreParams& P, int r, double& acc) {
  const uint4 f = __ldg(static_cast<const uint4*>(P.fast) + r);
  if ((f.x >> 31) != 0u) return false;          // scored by the list-driven phases: several records / different keys
  if (((f.x >> 30) & 1u) != 0u) return true;    // a mate without any record: no pair term, the value stands
  const uint4* __restrict__ comb = static_cast<const uint4*>(P.comb) + 4 * (size_t)(f.x & 0x3fffffffu);
  uint4 a1, a2, b1, b2;
  ldg256(comb, a1, a2);
  ldg256(comb + 2, b1, b2);
  const int4 te = __ldg(static_cast<const int4*>(P.tq) + f.w);
  const bool live1 = (a1.x & 0x7fffffffu) == P.epoch, live2 = (a2.x & 0x7fffffffu) == P.epoch;
  if (!live1 || !live2) return !live1 && !live2 ? true : false;   // (both stores hold the key or neither does)
  const int n1 = (int)b1.y, n2 = (int)b2.y;
  if (n1 != n2 || n1 > 2) return false;
  int4 o1 = make_int4((int)a1.y, 0, (int)a1.z, (int)a1.w), o2 = make_int4((int)a2.y, 0, (int)a2.z, (int)a2.w);   // {walk, -, cur_pos, skip_below}
  int4 p1 = o1, p2 = o2;
  if (n1 == 2) {
    p1 = ldg4(P.m[0].occ + b1.z + 1);   // {walk, seg, cur_pos, skip_below}
    p2 = ldg4(P.m[1].occ + b2.z + 1);
    if (p1.x == o1.x || p1.x != p2.x) return false;   // the key twice in ONE walk: distances between the occurrences matter
  }
  if (o1.x != o2.x) return false;
  const double t = __hiloint2double(te.y, te.x);
  const int pos1 = (int)f.y, pos2 = (int)f.z;
  if (wrap_add(pos1, o1.z) >= o1.w && wrap_add(pos2, o2.z) >= o2.w) acc = o1.x < P.n_erased ? __dsub_rn(acc, t) : __dadd_rn(acc, t);
  if (n1 == 2 && wrap_add(pos1, p1.z) >= p1.w && wrap_add(pos2, p2.z) >= p2.w) acc = p1.x < P.n_erased ? __dsub_rn(acc, t) : __dadd_rn(acc, t);
  return true;
}

// DELTA discovery + update: one thread per mate-1 record under a key of an erased/added walk; the first
// thread to stamp a read owns it and replays that read's subtract/add sequence.
__global__ void __launch_bounds__(kOvfBlock) paired_delta_kernel(const ScoreParams P) {
  tl_begin(P.timeline, kTlDelta);
  pdl_release();
  pdl_wait();
  const double2* log_tab = static_cast<const double2*>(P.log_tab);
  Acc sum = acc_zero();
  unsigned floored = 0;
  // the touched keys' range table in shared memory: every thread searches it
  constexpr int kTouchShared = 1024;
  __shared__ uint32_t s_prefix[kTouchShared + 1];
  __shared__ uint32_t s_begin[kTouchShared];
  const bool in_shared = P.n_touch <= kTouchShared;
  if (in_shared) {
    for (int t = threadIdx.x; t <= P.n_touch; t += blockDim.x) {
      s_prefix[t] = __ldg(P.touch_prefix + t);
      if (t < P.n_touch) s_begin[t] = P.touch[t].begin;
    }
    __syncthreads();
  }
  const uint32_t total = in_shared ? s_prefix[P.n_touch] : __ldg(P.touch_prefix + P.n_touch);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    int lo = 0, hi = P.n_touch;   // largest t with prefix[t] <= i
    uint32_t at;
    if (in_shared) {
      while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (s_prefix[mid] <= i) lo = mid; else hi = mid;
      }
      at = s_begin[lo] + (i - s_prefix[lo]);
    } else {
      while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(P.touch_prefix + mid) <= i) lo = mid; else hi = mid;
      }
      at = P.touch[lo].begin + (i - __ldg(P.touch_prefix + lo));
    }
    const int r = ldg4(P.arena1 + at).x;
    if (atomicExch(P.stamp + r, P.epoch) == P.epoch) continue;
    const double old = P.values[r];
    double acc = old;
    if ((P.fast && P.tq && !P.ev_keys && delta_fast(P, r, acc)) || paired_read_ordered(P, r, acc)) {
      P.values[r] = acc;
      if (P.delta_only) {   // same total length as the running total: swap this read's term in it
        const uint32_t ll = __ldg(P.lens + r);
        double pstar;
        long long qthr;
        term_consts(P, (ll & 0xffff) + (ll >> 16), pstar, qthr);
        acc_term_sub(sum, floored, log_tab, old, pstar, qthr);
        acc_term(sum, floored, log_tab, acc, pstar, qthr);
      }
    } else {
      push_overflow(P, r);
    }
  }
  if (P.delta_only) {
    block_accumulate(sum, floored, P.accum);
    finish_set_if_complete(P);
  }
  tl_end(P.timeline, kTlDelta);
}

// Many-placement pass: the reads the streaming / delta kernel listed because they need the enumeration order.
// full_mode 1: full evaluation (state from 0, terms summed, per-set finalize); 0: delta followed by the O(R) total pass;
// 2: delta-only evaluation (new term - old term into the running total, per-set finalize). In modes 1 and 2 the kernel
// before it has already published the set when it listed nothing (P.done). Mode 1 also runs on its own, submitted by the
// host after a chain without it ended with a pending line (launch_paired_tail).
__global__ void __launch_bounds__(kOvfBlock) paired_overflow_kernel(const ScoreParams P, int full_mode) {
  tl_begin(P.timeline, kTlOverflow);
  pdl_release();
  pdl_wait();
  if (full_mode && __ldcg(P.done)) {
    tl_end(P.timeline, kTlOverflow);
    return;
  }
  const double2* log_tab = static_cast<const double2*>(P.log_tab);
  Acc sum = acc_zero();
  unsigned floored = 0;
  const uint32_t n = min(*P.ovf_count, P.ovf_cap);
  for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
    const int r = (int)P.ovf_list[k];
    const double old = full_mode == 1 ? 0.0 : P.values[r];
    double acc = old;
    const uint32_t ll = __ldg(P.lens + r);
    if (paired_read_any(P, r, ll, acc)) P.values[r] = acc;
    if (full_mode) {
      double pstar;
      long long qthr;
      term_consts(P, (ll & 0xffff) + (ll >> 16), pstar, qthr);
      acc_term(sum, floored, log_tab, acc, pstar, qthr);
      if (full_mode == 2) acc_term_sub(sum, floored, log_tab, old, pstar, qthr);   // delta-only: the previous term leaves the running total
    }
  }
  if (full_mode) {
    block_accumulate(sum, floored, P.accum);
    finish_set(P);
  }
  tl_end(P.timeline, kTlOverflow);
}

// O(R) pass after a delta: GetTotalProb over the persistent probs (graph.cc:1495-1516).
__global__ void __launch_bounds__(kBlock) paired_total_kernel(const ScoreParams P) {
  tl_begin(P.timeline, kTlTotal);
  pdl_release();
  pdl_wait();
  Acc sum = acc_zero();
  unsigned floored = 0;
  const int stride = gridDim.x * blockDim.x;
  int r = blockIdx.x * blockDim.x + threadIdx.x;
  // software-pipelined like the full kernel: next read's state and lengths are in flight while this one's log runs
  bool have = r < P.n_reads;
  double v = 0.0;
  uint32_t ll = 0;
  if (have) { v = P.values[r]; ll = __ldg(P.lens + r); }
  while (have) {
    const int rn = r + stride;
    const bool have_next = rn < P.n_reads;
    double nv = 0.0;
    uint32_t nll = 0;
    if (have_next) { nv = P.values[rn]; nll = __ldg(P.lens + rn); }
    acc_read(P, sum, floored, v, (ll & 0xffff) + (ll >> 16));
    v = nv; ll = nll; r = rn; have = have_next;
  }
  block_accumulate(sum, floored, P.accum);
  finish_set(P);
  tl_end(P.timeline, kTlTotal);
}

// ---- single -------------------------------------------------------------------------------
// CalcScoreForPaths (graph.cc:1650-1743): placements of all walks pooled per read, de-duplicated on the
// global position, summed in enumeration order.
__device__ double single_sum(const ScoreParams& P, Plc* a, int n, int len) {
  sort_by_ord(a, n);
  const int m = dedup_positions(a, 0, n);
  double acc = 0.0;
  for (int x = 0; x < m; x++) acc = __dadd_rn(acc, align_prob(P.m[0], a[x].edor, len));
  return acc;
}

// One read through the register path (<= 2 live placements); false = needs the scratch path.
template <bool kCompact = false>
__device__ __forceinline__ bool single_read(const ScoreParams& P, int r, int len, double& acc) {
  Few a;
  scan_two<kCompact>(P.m[0], P.epoch, r, a);
  if (a.n > kFew) return false;
  acc = 0.0;
  const unsigned valid = order_few(a);   // all walks are one group here (walk ordinal 0): de-dup on the global position
#pragma unroll
  for (int x = 0; x < kFew; x++)
    if ((valid >> x) & 1u) acc = __dadd_rn(acc, align_prob(P.m[0], a.edor[x], len));
  return true;
}

// Tier 1: reads with at most one record (static) whose key occurs at most once in this evaluation.
__global__ void __launch_bounds__(kBlock) single_full_kernel(const ScoreParams P) {
  pdl_wait();
  pdl_release();   // after the wait: tier 2 starts without one (see launch_paired_full)
  Acc sum = acc_zero();
  unsigned floored = 0;
  const int4* first = static_cast<const int4*>(P.m[0].first);
  for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < P.n_reads; r += gridDim.x * blockDim.x) {
    const int4 rw = __ldg(first + r);
    const int len = (int)__ldg(P.lens + r);
    if (((rw.z >> 17) & 0x1fff) != 0) continue;   // several records: tier 2
    double acc = 0.0;
    if (rw.x >= 0) {
      const uint32_t ef = (uint32_t)ldg4(P.m[0].slots_a + rw.x).x;
      if ((ef & 0x7fffffffu) == P.epoch) {
        if (ef >> 31) {
          push_overflow(P, r);
          continue;
        }
        acc = __dadd_rn(acc, align_prob(P.m[0], rw.z, len));   // no skip rule for single reads (graph.cc:632-645)
      }
    }
    P.values[r] = acc;
    acc_read(P, sum, floored, acc, (uint32_t)len);
  }
  block_accumulate(sum, floored, P.accum);
}

__global__ void __launch_bounds__(kBlock) single_complex_kernel(const ScoreParams P) {
  pdl_release();   // no wait here, one at the end: same chain discipline as the paired streaming kernel
  Acc sum = acc_zero();
  unsigned floored = 0;
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < P.n_complex; k += gridDim.x * blockDim.x) {
    const int r = (int)__ldg(P.complex_list + k);
    const int len = (int)__ldg(P.clens + k);
    double acc;
    if (single_read<true>(P, k, len, acc)) {
      P.values[r] = acc;
      acc_read(P, sum, floored, acc, (uint32_t)len);
    } else {
      push_overflow(P, r);
    }
  }
  pdl_wait();
  block_accumulate(sum, floored, P.accum);
}

__global__ void __launch_bounds__(kOvfBlock) single_overflow_kernel(const ScoreParams P) {
  pdl_release();
  pdl_wait();
  Acc sum = acc_zero();
  unsigned floored = 0;
  const uint32_t n = min(*P.ovf_count, P.ovf_cap);
  for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
    const int r = (int)P.ovf_list[k];
    const int n1 = gather_short(P.m[0], P.epoch, r, nullptr);
    const unsigned long long base = atomicAdd(P.scratch_cursor, (unsigned long long)n1);
    const int len = (int)__ldg(P.lens + r);
    double acc = 0.0;
    if (base + n1 > P.scratch_cap) {
      atomicOr(P.error_flag, 2u);
    } else {
      Plc* a = P.scratch + base;
      gather_short(P.m[0], P.epoch, r, a);
      acc = single_sum(P, a, n1, len);
    }
    P.values[r] = acc;
    acc_read(P, sum, floored, acc, (uint32_t)len);
  }
  block_accumulate(sum, floored, P.accum);
  finish_set(P);
}

// ---- pacbio (log space; logdouble.hpp) -----------------------------------------------------
// logdouble::operator+= (logdouble.hpp:21-31): -inf is the additive identity, otherwise
// max + log1p(exp(min - max)).
__device__ __forceinline__ double lse_add(double acc, double v) {
  if (isinf(acc) && acc < 0) return v;
  if (isinf(v) && v < 0) return acc;
  const double hi = fmax(acc, v), lo = fmin(acc, v);
  return __dadd_rn(hi, log1p(exp(__dsub_rn(lo, hi))));
}

// Warp-shuffle log-sum-exp (order-free variant used for very long placement lists): max-reduce, then
// sum of exp(v - max) in the warp, then one log.
__device__ __forceinline__ double warp_lse(double v) {
  double m = v;
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, off));
  if (isinf(m) && m < 0) return m;
  double s = exp(__dsub_rn(v, m));
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) s = __dadd_rn(s, __shfl_xor_sync(0xffffffffu, s, off));
  return __dadd_rn(m, log(s));
}

__device__ __forceinline__ double pacbio_floor(const ScoreParams& P, double v, int len, unsigned& floored) {
  const double fl = __dadd_rn(P.floor_a, __dmul_rn(P.floor_b, (double)len));   // graph.cc:3075-3076
  if (v < fl) { floored++; v = fl; }
  return v;
}

__global__ void __launch_bounds__(kBlock) pacbio_full_kernel(const ScoreParams P) {
  pdl_release();
  pdl_wait();
  Acc sum = acc_zero();
  unsigned floored = 0;
  for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < P.n_reads; r += gridDim.x * blockDim.x) {
    PlcLong a[kCapLong];
    int n = 0;
    for_each_long(P.m[0], P.epoch, r, [&](const int4& o, const int4& rw, int idx) {
      if (n < kCapLong) {
        a[n].ord = ((unsigned long long)(uint32_t)o.y << 32) | (uint32_t)idx;
        a[n].logprob = __hiloint2double(rw.w, rw.z);
      }
      n++;
    });
    if (n > kCapLong) {
      push_overflow(P, r);
      continue;
    }
    double acc = -INFINITY;
    if (n == 1) {
      acc = a[0].logprob;
    } else if (n > 1) {
      sort_by_ord(a, n);
      for (int x = 0; x < n; x++) acc = lse_add(acc, a[x].logprob);
    }
    P.values[r] = acc;
    acc_add_log(sum, pacbio_floor(P, acc, (int)__ldg(P.lens + r), floored));
  }
  block_accumulate(sum, floored, P.accum);
}

// One WARP per many-placement read: lanes fold a strided share of the read's records sequentially and the 32
// partial log-sums are combined with the warp-shuffle LSE (order-free; within the 1e-12 per-read budget).
__global__ void __launch_bounds__(kOvfBlock) pacbio_overflow_kernel(const ScoreParams P) {
  pdl_release();
  pdl_wait();
  Acc sum = acc_zero();
  unsigned floored = 0;
  const uint32_t n = min(*P.ovf_count, P.ovf_cap);
  const int lane = threadIdx.x & 31, n_warps = (gridDim.x * blockDim.x) >> 5;
  for (uint32_t k = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; k < n; k += n_warps) {
    const int r = (int)P.ovf_list[k];
    const MateView& mv = P.m[0];
    const uint32_t b = __ldg(mv.rowptr + r), e = __ldg(mv.rowptr + r + 1);
    const RowLong* rows = static_cast<const RowLong*>(mv.rows);
    double part = -INFINITY;
    for (uint32_t i = b + lane; i < e; i += 32) {
      const int4 rw = ldg4(rows + i);
      if (((uint32_t)ldg4(mv.slots_a + rw.x).x & 0x7fffffffu) != P.epoch) continue;
      const int n_occ = ldg4(mv.slots_b + rw.x).y;
      const double lp = __hiloint2double(rw.w, rw.z);
      for (int t = 0; t < n_occ; t++) part = lse_add(part, lp);   // same record under n_occ live lookups
    }
    const double acc = warp_lse(part);
    if (lane == 0) {
      P.values[r] = acc;
      acc_add_log(sum, pacbio_floor(P, acc, (int)__ldg(P.lens + r), floored));
    }
  }
  block_accumulate(sum, floored, P.accum);
  finish_set(P);
}

// ---- batched candidate evaluation (BASELINE config 5) ------------------------------------------------
// Candidate c replaces a few walks of the last evaluated walk set. Its score is
//     sum over ALL reads of term(base value, L_c)  +  sum over reads touched by c of [term(new value, L_c) - term(base value, L_c)]
// with exactly the per-read arithmetic of a normal evaluation; all sums are exact integers, so the result is the
// double gaml_calc_prob would return for the candidate's walk set — without touching the state.
// First sum, ONE pass over the base state for all the batch's total lengths (SURVEY §7.4.3): the lengths are sorted
// ascending, so a read's floor test p < pstar(L_j) is monotone in j — it is not floored below k = its first floored
// index and floored from k on. sum_j = sum over all reads of qthr + sum over reads with k > j of (Q - qthr), i.e. a
// histogram over k and a suffix sum (batch_prefix_kernel). The two ends of the range (never floored: nearly every placed
// read; always floored: unplaced reads) are kept in registers, the rest goes through shared-memory bins.
struct TermAt { long long q; int floored; int odd; };   // odd: 1 = -inf, 2 = nan (q = 0 then)
__device__ __forceinline__ TermAt term_at(const double2* log_tab, double p, double pstar, long long qthr) {
  if (p < pstar) return TermAt{qthr, 1, 0};
  const double lg = table_log(log_tab, p);
  if (fabs(lg) < kFixLimit) return TermAt{__double2ll_rn(lg * kFixScale), 0, 0};
  return TermAt{0ll, 0, lg == -INFINITY ? 1 : 2};
}

constexpr int kBatchMaxLen = 1024;   // distinct total lengths one base pass handles (longer batches: several passes)
__global__ void __launch_bounds__(kBlock) batch_base_kernel(const ScoreParams P, const BatchParams B, int j0, int nb, size_t hist_off) {
  __shared__ unsigned long long bins[(kBatchMaxLen + 1) * kBatchBin];
  for (int i = threadIdx.x; i < (nb + 1) * kBatchBin; i += blockDim.x) bins[i] = 0ull;
  __syncthreads();
  const double2* log_tab = static_cast<const double2*>(P.log_tab);
  // registers: [0] bin 0 (floored at every length), [1] bin nb (floored at none); all reads' qthr
  unsigned long long lo[2] = {0ull, 0ull}, cnt[2] = {0ull, 0ull}, ninf[2] = {0ull, 0ull}, bad[2] = {0ull, 0ull};
  long long hi[2] = {0ll, 0ll};
  Acc all_thr = acc_zero();
  for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < P.n_reads; r += gridDim.x * blockDim.x) {
    const uint32_t ll = __ldg(P.lens + r);
    const int cls = __ldg(B.len_class + (ll & 0xffff) + (ll >> 16));
    const double* row = B.pstar + (size_t)cls * B.n_len + j0;
    const long long qthr = __ldg(B.qthr_cls + cls);
    const double p = P.values[r];
    acc_add_q(all_thr, qthr);
    int k;   // first j (relative to j0) with p < pstar_j; NaN compares false everywhere -> nb, like the per-length test
    if (!(p < __ldg(row + nb - 1))) k = nb;
    else if (p < __ldg(row)) k = 0;
    else {
      int a = 0, b = nb - 1;   // row[a] <= p < row[b]
      while (b - a > 1) {
        const int mid = (a + b) >> 1;
        if (p < __ldg(row + mid)) b = mid; else a = mid;
      }
      k = b;
    }
    long long dq = -qthr;
    int odd = 0;
    if (k > 0) {   // a logarithm term at some length
      const double lg = table_log(log_tab, p);
      if (fabs(lg) < kFixLimit) dq = __double2ll_rn(lg * kFixScale) - qthr;
      else odd = lg == -INFINITY ? 1 : 2;
    } else {
      dq = 0;      // never used: no length index lies below bin 0
    }
    if (k == 0 || k == nb) {
      const int s = k == 0 ? 0 : 1;
      lo[s] += (unsigned long long)(uint32_t)dq;
      hi[s] += dq >> 32;
      cnt[s]++;
      ninf[s] += odd == 1;
      bad[s] += odd == 2;
    } else {
      unsigned long long* bin = bins + (size_t)k * kBatchBin;
      atomicAdd(bin, (unsigned long long)(uint32_t)dq);
      atomicAdd(bin + 1, (unsigned long long)(dq >> 32));
      atomicAdd(bin + 2, 1ull);
      if (odd == 1) atomicAdd(bin + 3, 1ull);
      if (odd == 2) atomicAdd(bin + 4, 1ull);
    }
  }
#pragma unroll
  for (int s = 0; s < 2; s++) {
    unsigned long long* bin = bins + (size_t)(s == 0 ? 0 : nb) * kBatchBin;
    if (cnt[s]) {
      atomicAdd(bin, lo[s]);
      atomicAdd(bin + 1, (unsigned long long)hi[s]);
      atomicAdd(bin + 2, cnt[s]);
      if (ninf[s]) atomicAdd(bin + 3, ninf[s]);
      if (bad[s]) atomicAdd(bin + 4, bad[s]);
    }
  }
  __syncthreads();
  unsigned long long* out = B.hist + hist_off * kBatchBin;   // chunks of lengths keep their own nb + 1 bins: see launch_batch
  for (int i = threadIdx.x; i < (nb + 1) * kBatchBin; i += blockDim.x)
    if (bins[i]) atomicAdd(out + i, bins[i]);
  // sum of qthr over all reads: the same for every length; accumulated next to the first bin set only
  if (j0 == 0) block_accumulate(all_thr, 0u, B.accum_len + (size_t)B.n_len * kAccumStride);
}

// Suffix sums of the histogram: accum_len[j] = {low, high 64 bits of sum_all qthr + sum_{k > j} (Q - qthr), floored = reads
// with k <= j, -inf / nan terms of the reads with k > j}. One block per chunk of lengths, bins [hist_off, hist_off + nb].
__global__ void __launch_bounds__(kBatchMaxLen) batch_prefix_kernel(const BatchParams B, int j0, int nb, size_t hist_off) {
  __shared__ unsigned long long bins[(kBatchMaxLen + 1) * kBatchBin];
  const unsigned long long* h = B.hist + hist_off * kBatchBin;
  for (int i = threadIdx.x; i < (nb + 1) * kBatchBin; i += blockDim.x) bins[i] = h[i];
  __syncthreads();
  const int j = threadIdx.x;
  if (j >= nb) return;
  const unsigned long long* base = B.accum_len + (size_t)B.n_len * kAccumStride;   // limbs of sum_all qthr
  unsigned __int128 x = 0;
  for (int t = 0; t < 4; t++) x += (unsigned __int128)base[t] << (32 * t);
  __int128 v = (__int128)x;
  unsigned long long floored = 0, ninf = 0, bad = 0;
  for (int k = 0; k <= nb; k++) {
    const unsigned long long* bin = bins + (size_t)k * kBatchBin;
    if (k > j) {
      v += (__int128)bin[0] + ((__int128)(long long)bin[1] << 32);
      ninf += bin[3];
      bad += bin[4];
    } else {
      floored += bin[2];
    }
  }
  unsigned long long* o = B.accum_len + (size_t)(j0 + j) * kAccumStride;
  o[0] = (unsigned long long)(unsigned __int128)v;
  o[1] = (unsigned long long)((unsigned __int128)v >> 64);
  o[2] = floored;
  o[3] = ninf;
  o[4] = bad;
}

// Second sum: a block per candidate (per kBatchSlice-record slice of a large one) over the mate-1 records under the keys the candidate touches. The candidate's own
// tables — touched ranges, sorted key ids and slot words of both mates — are staged in shared memory once, so a record
// costs its arena word, the read's FastPair, its value and one term-table entry; the thread whose record is the FIRST
// touched record of its read owns the read (no claim words: different candidates share reads in the same launch), and a
// fast read has only the one. The candidate's sums are reduced in the block and stored, no global atomics.
constexpr int kCandKeys = 192;     // keys per mate staged in shared memory (more: looked up in global memory)
constexpr int kCandRanges = 256;
__global__ void __launch_bounds__(kBlock) batch_touch_kernel(const ScoreParams P, const BatchParams B) {
  if ((int)blockIdx.x >= B.n_blocks) return;
  const Int2 blk = B.blocks[blockIdx.x];   // {candidate, first record of this block's slice}
  const int c = blk.x;
  const BatchCand cd = B.cands[c];
  const double2* log_tab = static_cast<const double2*>(P.log_tab);
  __shared__ int s_keys[2][kCandKeys];
  __shared__ int4 s_a[2][kCandKeys], s_b[2][kCandKeys];
  __shared__ uint32_t s_prefix[kCandRanges + 1], s_begin[kCandRanges];
  __shared__ long long s_acc[4];
  const bool keys_in_shared = cd.key_count[0] <= kCandKeys && cd.key_count[1] <= kCandKeys;
  const bool ranges_in_shared = cd.range_count <= kCandRanges;
  if (threadIdx.x < 4) s_acc[threadIdx.x] = 0;
  if (keys_in_shared) {
    for (int m = 0; m < 2; m++)
      for (int k = threadIdx.x; k < cd.key_count[m]; k += blockDim.x) {
        s_keys[m][k] = __ldg(B.keys[m] + cd.key_begin[m] + k);
        s_a[m][k] = __ldg(static_cast<const int4*>(B.slot_a[m]) + cd.key_begin[m] + k);
        s_b[m][k] = __ldg(static_cast<const int4*>(B.slot_b[m]) + cd.key_begin[m] + k);
      }
  }
  const uint32_t p0 = __ldg(B.range_prefix + cd.range_begin);
  if (ranges_in_shared)
    for (int t = threadIdx.x; t <= cd.range_count; t += blockDim.x) {
      s_prefix[t] = __ldg(B.range_prefix + cd.range_begin + t) - p0;
      if (t < cd.range_count) s_begin[t] = B.ranges[cd.range_begin + t].begin;
    }
  __syncthreads();
  const uint32_t cand_total = __ldg(B.range_prefix + cd.range_begin + cd.range_count) - p0;
  const uint32_t slice_begin = (uint32_t)blk.y, total = min(cand_total, slice_begin + (uint32_t)kBatchSlice);
  CandLookup lk0{B.keys[0] + cd.key_begin[0], cd.key_count[0], static_cast<const int4*>(B.slot_a[0]) + cd.key_begin[0],
                 static_cast<const int4*>(B.slot_b[0]) + cd.key_begin[0], B.occ[0]};
  CandLookup lk1{B.keys[1] + cd.key_begin[1], cd.key_count[1], static_cast<const int4*>(B.slot_a[1]) + cd.key_begin[1],
                 static_cast<const int4*>(B.slot_b[1]) + cd.key_begin[1], B.occ[1]};
  if (keys_in_shared) {   // the general replay searches the staged copies too
    lk0.keys = s_keys[0]; lk0.a = s_a[0]; lk0.b = s_b[0];
    lk1.keys = s_keys[1]; lk1.a = s_a[1]; lk1.b = s_b[1];
  }
  auto find_key = [&](int m, int key) {   // index of `key` among the candidate's keys of mate m, or -1
    const int n = cd.key_count[m];
    int l = 0, h = n;
    if (keys_in_shared) {
      while (l < h) { const int mid = (l + h) >> 1; if (s_keys[m][mid] < key) l = mid + 1; else h = mid; }
      return (l < n && s_keys[m][l] == key) ? l : -1;
    }
    const int* keys = B.keys[m] + cd.key_begin[m];
    while (l < h) { const int mid = (l + h) >> 1; if (__ldg(keys + mid) < key) l = mid + 1; else h = mid; }
    return (l < n && __ldg(keys + l) == key) ? l : -1;
  };
  long long sum_lo = 0, sum_hi = 0, d_floored = 0, n_bad = 0;
  auto locate = [&](uint32_t i, uint32_t& ai) {   // i-th touched record of the candidate -> arena index
    int lo = 0, hi = cd.range_count;   // largest t with prefix[t] <= i
    if (ranges_in_shared) {
      while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (s_prefix[mid] <= i) lo = mid; else hi = mid; }
      ai = s_begin[lo] + (i - s_prefix[lo]);
    } else {
      const uint32_t* pre = B.range_prefix + cd.range_begin;
      while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (__ldg(pre + mid) - p0 <= i) lo = mid; else hi = mid; }
      ai = B.ranges[cd.range_begin + lo].begin + (i - (__ldg(pre + lo) - p0));
    }
  };
  auto account = [&](int r, double v0, double v1) {   // the read's term at the candidate's total length: new - old
    if (v1 == v0) return;   // bit-identical value: identical term
    const uint32_t ll = __ldg(P.lens + r);
    const int cls = __ldg(B.len_class + (ll & 0xffff) + (ll >> 16));
    const double pstar = __ldg(B.pstar + (size_t)cls * B.n_len + cd.len_index);
    const long long qthr = __ldg(B.qthr_cls + cls);
    const TermAt t0 = term_at(log_tab, v0, pstar, qthr), t1 = term_at(log_tab, v1, pstar, qthr);
    if (!t0.odd && !t1.odd) {
      const long long dq = t1.q - t0.q;   // |q| < 2^62: no overflow
      sum_lo += (long long)(uint32_t)dq;   // low 32 bits
      sum_hi += dq >> 32;                  // high part, signed
    } else {
      n_bad++;   // non-finite term: reported as nan
    }
    d_floored += t1.floored - t0.floored;
  };
  // Chunks of the candidate's records, two passes each: (A) every record — fast reads are finished on the spot, the others
  // are queued; (B) the queue, densely: the general replay is ~10x a fast read's work, and taken lane by lane inside pass A
  // it would make every warp pay for it on every trip.
  constexpr int kChunk = 2048;
  __shared__ uint32_t s_queue[kChunk];
  __shared__ int s_qn;
  const bool fast_path = P.fast && P.tq && B.partner12;
  for (uint32_t chunk = slice_begin; chunk < total; chunk += kChunk) {
    if (threadIdx.x == 0) s_qn = 0;
    __syncthreads();
    const uint32_t chunk_end = min(total, chunk + (uint32_t)kChunk);
    for (uint32_t i = chunk + threadIdx.x; i < chunk_end; i += blockDim.x) {
      uint32_t ai;
      locate(i, ai);
      const int r = ldg4(P.arena1 + ai).x;
      bool done = false;
      if (fast_path) {
        // a FAST read (one record per mate under one key, term resolved at commit — FastPair): its only mate-1 record is
        // the one this thread holds, and the replay is "T leaves / enters per occurrence of the key in the candidate's
        // erased / added walks" exactly like delta_fast, from the candidate's own key tables
        const uint4 f = __ldg(static_cast<const uint4*>(P.fast) + r);
        if ((f.x >> 31) == 0u) {
          if (((f.x >> 30) & 1u) != 0u) continue;   // a mate without any record: no pair term, nothing changes
          const int k1 = (int)(f.x & 0x3fffffffu), k2 = __ldg(B.partner12 + k1);
          const int i1 = find_key(0, k1), i2 = k2 >= 0 ? find_key(1, k2) : -1;
          if (i1 < 0 || i2 < 0) continue;   // the key is not in this candidate's walks for one of the mates: no pair term changes
          const int4 a1 = lk0.a[i1], b1 = lk0.b[i1], a2 = lk1.a[i2], b2 = lk1.b[i2];
          if (b1.y == b2.y && b1.y <= 2) {
            int4 o1 = make_int4(a1.y, 0, a1.z, a1.w), o2 = make_int4(a2.y, 0, a2.z, a2.w);   // {walk, -, cur_pos, skip_below}
            int4 q1 = o1, q2 = o2;
            bool ok = o1.x == o2.x;
            if (b1.y == 2) {
              q1 = ldg4(lk0.occ + b1.z + 1);
              q2 = ldg4(lk1.occ + b2.z + 1);
              ok = ok && q1.x != o1.x && q1.x == q2.x;   // (the key twice in ONE walk: the general path)
            }
            if (ok) {
              const int4 te = __ldg(static_cast<const int4*>(P.tq) + f.w);
              const double t = __hiloint2double(te.y, te.x);
              const int pos1 = (int)f.y, pos2 = (int)f.z;
              const double v0 = P.values[r];
              double v1 = v0;
              if (wrap_add(pos1, o1.z) >= o1.w && wrap_add(pos2, o2.z) >= o2.w) v1 = o1.x < cd.n_erased ? __dsub_rn(v1, t) : __dadd_rn(v1, t);
              if (b1.y == 2 && wrap_add(pos1, q1.z) >= q1.w && wrap_add(pos2, q2.z) >= q2.w)
                v1 = q1.x < cd.n_erased ? __dsub_rn(v1, t) : __dadd_rn(v1, t);
              account(r, v0, v1);
              done = true;
            }
          }
        }
      }
      if (!done) s_queue[atomicAdd(&s_qn, 1)] = i;
    }
    __syncthreads();
    const int qn = s_qn;
    for (int q = threadIdx.x; q < qn; q += blockDim.x) {
      uint32_t ai;
      locate(s_queue[q], ai);
      const int r = ldg4(P.arena1 + ai).x;
      {   // ownership: is there an earlier record of this read under a key of this candidate?
        const MateView& mv = P.m[0];
        const int4 f = ldg4(static_cast<const int4*>(mv.first) + r);
        int cnt = (f.z >> 16) & 0x3fff;
        const uint32_t base = (uint32_t)f.w;
        if (cnt == 0x3fff) cnt = (int)(__ldg(mv.rowptr + r + 1) - base);
        const RowShort* rows = static_cast<const RowShort*>(mv.rows);
        bool owner = true;
        for (int k = 0; k < cnt; k++) {
          const int4 rw = ldg4(rows + base + k);
          if ((uint32_t)rw.w >= ai) break;   // rows are in arena order
          if (find_key(0, rw.x) >= 0) { owner = false; break; }
        }
        if (!owner) continue;
      }
      const double v0 = P.values[r];
      double v1 = v0;
      if (!paired_read_with(P, lk0, lk1, r, v1, cd.n_erased)) {
        // many-placement read: same replay from a scratch allocation, inline (rare)
        const int n1 = gather_short(P.m[0], lk0, r, nullptr), n2 = gather_short(P.m[1], lk1, r, nullptr);
        const unsigned long long at = atomicAdd(P.scratch_cursor, (unsigned long long)(n1 + n2));
        if (at + n1 + n2 > P.scratch_cap) {
          atomicOr(P.error_flag, 2u);
          continue;
        }
        Plc* a = P.scratch + at;
        Plc* b = a + n1;
        gather_short(P.m[0], lk0, r, a);
        gather_short(P.m[1], lk1, r, b);
        const uint32_t ll = __ldg(P.lens + r);
        v1 = apply_pairs(P, a, n1, b, n2, ll & 0xffff, ll >> 16, v0, cd.n_erased);
      }
      account(r, v0, v1);
    }
    __syncthreads();
  }
  if (sum_lo) atomicAdd(reinterpret_cast<unsigned long long*>(&s_acc[0]), (unsigned long long)sum_lo);
  if (sum_hi) atomicAdd(reinterpret_cast<unsigned long long*>(&s_acc[1]), (unsigned long long)sum_hi);
  if (d_floored) atomicAdd(reinterpret_cast<unsigned long long*>(&s_acc[2]), (unsigned long long)d_floored);
  if (n_bad) atomicAdd(reinterpret_cast<unsigned long long*>(&s_acc[3]), (unsigned long long)n_bad);
  __syncthreads();
  if (threadIdx.x < 4 && s_acc[threadIdx.x])   // (a candidate with many touched records is spread over several blocks)
    atomicAdd(reinterpret_cast<unsigned long long*>(B.accum_cand + (size_t)c * 4 + threadIdx.x), (unsigned long long)s_acc[threadIdx.x]);
}

// out[c] = {integer part, 2^-40 units, floored, -inf terms, nan terms, flags} like finalize_kernel.
__global__ void batch_finalize_kernel(const BatchParams B, double* out, const uint32_t* error_flag, long long n_reads) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= B.n_cand) return;
  const int j = B.cands[c].len_index;
  const unsigned long long* a = B.accum_len + (size_t)j * kAccumStride;
  const long long* dl = B.accum_cand + (size_t)c * 4;
  const long long floored = (long long)a[2] + dl[2], ninf = (long long)a[3], bad = (long long)a[4] + dl[3];
  __int128 v = (__int128)(((unsigned __int128)a[1] << 64) | (unsigned __int128)a[0]) + (__int128)dl[0] + ((__int128)dl[1] << 32);
  v -= (__int128)(n_reads - floored - ninf - bad) * (__int128)B.ql[j];   // the - FIX(log 2L) part of every logarithm term (publish_set)
  const long long ip = (long long)(v >> 40);
  const unsigned long long fr = (unsigned long long)((unsigned __int128)v & (((unsigned __int128)1 << 40) - 1));
  double* o = out + (size_t)c * kOutStride;
  o[0] = (double)ip;
  o[1] = (double)fr;
  o[2] = (double)floored;
  o[3] = (double)ninf;
  o[4] = (double)bad;
  o[5] = (double)(*error_flag);
}

// ---- coverage-gap penalty of paired sets (graph.cc:1893-1919) ----------------------------------------
// Events sorted by (walk, position, type): contig starts (type 1, host supplied) and covered positions (type 3).
// bad_bases(walk) = sum over type-3 events whose distance to the PREVIOUS event of the walk exceeds `step`, when that
// previous event is also type 3 (or the walk has no previous event) and the position is further than
// insert_mean + 5 insert_std from the last contig start. Every event only looks at its predecessor, so the sweep is
// one independent thread per event after the sort.
__global__ void coverage_sweep_kernel(const unsigned long long* keys, unsigned n, const int* cs_begin, const int* cs,
                                      double step, double min_from_start, int* bad) {
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const unsigned long long k = keys[i];
    if (k == ~0ull || !(k & 1ull)) continue;   // padding or a contig start
    const int walk = (int)(k >> 33);
    const int pos = (int)(((uint32_t)(k >> 1)) ^ 0x80000000u);
    int prev_pos = 0, prev_type = -1;
    if (i > 0) {
      const unsigned long long p = keys[i - 1];
      if ((int)(p >> 33) == walk) {
        prev_pos = (int)(((uint32_t)(p >> 1)) ^ 0x80000000u);
        prev_type = (p & 1ull) ? 3 : 1;
      }
    }
    int last_begin = 0;
    for (int t = cs_begin[walk]; t < cs_begin[walk + 1]; t++) {   // contig starts of the walk, ascending (few)
      if (cs[t] <= pos) last_begin = cs[t]; else break;
    }
    if ((double)(pos - prev_pos) > step && (prev_type == 3 || prev_type < 0) && (double)(pos - last_begin) > min_from_start)
      atomicAdd(bad + walk, pos - prev_pos);
  }
}

// ---- PacBio coverage penalty (CalcScoreForPacbio, graph.cc:3197-3250) --------------------------------------------
// Per walk the reference sorts interval events — an artificial interval [-1000, 2000), one interval per node, one per
// alignment at least as probable as its read's minimum (graph.h:478) — and sweeps them with a multiset of open starts;
// after each event: good_start = min(earliest open start + step, next event, len - 250), and the stretch from
// max(2500, event) to good_start counts as bad. Only the LAST event of a position can contribute (for the others the
// next event is at the same position), and at that point the multiset holds exactly the intervals with
// start <= x < end — so the sweep needs no order inside a position and no multiset: sort the intervals of all walks by
// (walk, start), take the running maximum of their ends per walk, and the earliest-started interval still open at x is
// the first one whose running maximum exceeds x (binary search), if it has started.
__device__ __forceinline__ unsigned long long pb_key(int walk, int pos) {
  return ((unsigned long long)(uint32_t)walk << 32) | (unsigned long long)((uint32_t)pos ^ 0x80000000u);
}
__device__ __forceinline__ int pb_key_pos(unsigned long long k) { return (int)((uint32_t)k ^ 0x80000000u); }

__global__ void pacbio_cov_emit_kernel(const PbCovParams C) {
  const uint32_t total = (uint32_t)C.n_seed + __ldg(C.occ_prefix + C.n_occ);
  for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < total; q += gridDim.x * blockDim.x) {
    int walk, start, end;
    if (q < (uint32_t)C.n_seed) {
      const int4 sd = ldg4(static_cast<const int4*>(C.seeds) + q);   // {walk, start, end, -}: the artificial interval and the nodes
      walk = sd.x; start = sd.y; end = sd.z;
    } else {
      const uint32_t t = q - (uint32_t)C.n_seed;
      int lo = 0, hi = C.n_occ;   // largest o with prefix[o] <= t
      while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(C.occ_prefix + mid) <= t) lo = mid; else hi = mid;
      }
      const int4 oc = ldg4(static_cast<const int4*>(C.occ) + lo);   // {walk, offset of the key's first node in the walk, arena range begin, count}
      const uint32_t rec = (uint32_t)oc.z + (t - __ldg(C.occ_prefix + lo));
      const ArenaLong al = C.arena[rec];
      const double len = (double)__ldg(C.lens + al.read);
      const double min_lp = __dadd_rn(__dmul_rn(C.log_mismatch, __dmul_rn(len, 0.25)), __dmul_rn(C.log_match, __dmul_rn(len, 0.75)));
      if (al.logprob < min_lp) continue;   // graph.cc:3215
      const int2 be = static_cast<const int2*>(C.arena_pos)[rec];
      walk = oc.x; start = oc.y + be.x; end = oc.y + be.y;
    }
    const uint32_t slot = atomicAdd(C.count, 1u);
    if (slot >= C.cap) { atomicOr(C.error_flag, 4u); continue; }
    C.ikey[slot] = pb_key(walk, start);
    C.iend[slot] = end;
    C.pkey[2 * slot] = pb_key(walk, start);
    C.pkey[2 * slot + 1] = pb_key(walk, end);
  }
}

// (walk, running maximum of the interval ends) packed for a segmented inclusive max scan
__global__ void pacbio_cov_pack_kernel(const unsigned long long* ikey, const int* iend, unsigned long long* packed, uint32_t n) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) packed[i] = (ikey[i] & 0xffffffff00000000ull) | (unsigned long long)((uint32_t)iend[i] ^ 0x80000000u);
}
struct PbSegMax {
  __device__ __forceinline__ unsigned long long operator()(unsigned long long a, unsigned long long b) const {
    if ((a >> 32) != (b >> 32)) return b;
    return (uint32_t)a > (uint32_t)b ? a : b;
  }
};

__global__ void pacbio_cov_sweep_kernel(const unsigned long long* pkey, const unsigned long long* ikey, const unsigned long long* run_max,
                                        const uint32_t* count, uint32_t cap, const int* walk_len, double step, int* bad) {
  const uint32_t n_int = min(*count, cap), n_pos = 2 * n_int;
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n_pos; j += gridDim.x * blockDim.x) {
    const unsigned long long k = pkey[j];
    const int walk = (int)(k >> 32), x = pb_key_pos(k);
    bool has_next = false;
    int next_x = 0;
    if (j + 1 < n_pos) {
      const unsigned long long kn = pkey[j + 1];
      if ((int)(kn >> 32) == walk) {
        has_next = true;
        next_x = pb_key_pos(kn);
      }
    }
    if (has_next && next_x == x) continue;   // not the last event of this position
    // earliest-started interval of this walk that is still open after position x
    uint32_t lo = 0, hi = n_int;             // first interval with key >= (walk, -inf)
    const unsigned long long wk = (unsigned long long)(uint32_t)walk << 32;
    while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (ikey[mid] < wk) lo = mid + 1; else hi = mid; }
    const uint32_t seg_lo = lo;
    hi = n_int;                              // first interval of a later walk
    while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if ((ikey[mid] >> 32) <= (unsigned long long)(uint32_t)walk) lo = mid + 1; else hi = mid; }
    const uint32_t seg_hi = lo;
    uint32_t a = seg_lo, b = seg_hi;         // first interval whose running maximum of ends exceeds x
    while (a < b) {
      const uint32_t mid = (a + b) >> 1;
      if ((int)((uint32_t)run_max[mid] ^ 0x80000000u) > x) b = mid; else a = mid + 1;
    }
    const int tl = walk_len[walk];
    int good_start = tl - 250;
    if (a < seg_hi && pb_key_pos(ikey[a]) <= x) good_start = (int)((double)pb_key_pos(ikey[a]) + step);
    if (has_next) good_start = min(next_x, good_start);
    good_start = min(good_start, tl - 250);
    const int from = max(2500, x);
    if (good_start > from) atomicAdd(bad, good_start - from);
  }
}

// ---- PacBio alignment probability (PacbioReadSet::AligmentProbability, graph.cc:2175-2297) -----------------------
// Forward DP in log space over the cells around an alignment's CIGAR path: cell(row, col) = the probability of
// generating the read's first `col` bases from the walk's bases up to `row`, summed over the three predecessors
// (diagonal: match/mismatch, up: walk base against a gap, left: gap against a read base); the result is the sum of the
// cells in the read's last column.
// The reference lists the cells — (0,0), a block in front of an alignment that starts with insertions, the path, a
// block behind one that ends with insertions — fills every row between its smallest and largest listed column
// (Uniquify, graph.cc:2150-2173) and widens everything by the band in both directions (graph.cc:2210-2222). Here one
// thread per alignment walks the CIGAR ONCE, `band` rows ahead of the DP, keeping the column ranges of the 2*band+1
// path rows that reach the current DP row in a ring: nothing per row is prepared on the host or stored. Rows and
// columns run in the reference's order — the additions of the log-sum-exp chain are not associative, so the order
// is part of the result — with the previous and the current row in a per-thread scratch strip (L1/L2 resident).
// Compute bound: up to three exp + log1p per cell.
struct CigarWalk {   // yields the column range of the path's cells row by row
  const int32_t* len;
  const unsigned char* chr;
  int n_ops, k, rem, col;
  __device__ __forceinline__ void norm() {
    while (k < n_ops && rem == 0) {
      k++;
      if (k < n_ops) rem = len[k];
    }
  }
  __device__ __forceinline__ void start(const int32_t* l, const unsigned char* c, int n) {
    len = l; chr = c; n_ops = n; k = 0; col = 0;
    rem = n > 0 ? l[0] : 0;
    norm();
  }
  __device__ __forceinline__ void insertions() {
    while (k < n_ops && chr[k] == 'I') { col += rem; rem = 0; norm(); }
  }
  // row 0: cell (0,0) and the leading insertions; row > 0: one M or D step into the row, then insertions
  __device__ __forceinline__ bool row(int r, int& lo, int& hi) {
    if (r > 0) {
      if (k >= n_ops) return false;
      if (chr[k] == 'M') col++;
      rem--;
      norm();
    }
    lo = col;
    insertions();
    hi = col;
    return true;
  }
};

__global__ void __launch_bounds__(128) pacbio_alnprob_kernel(const AlnProbParams A) {
  const double ninf = -INFINITY;
  const int B = A.band;
  constexpr int kRing = 2 * kAlnMaxBand + 1;
  for (long long a = blockIdx.x * (long long)blockDim.x + threadIdx.x; a < A.n; a += (long long)gridDim.x * blockDim.x) {
    const AlnMeta m = A.meta[a];
    const unsigned char* s1 = A.s1 + m.s1_off;
    const unsigned char* s2 = A.s2 + m.s2_off;
    double* prev = A.scratch + m.scratch_off;
    double* cur = prev + m.width;
    const int row_min = m.bl > 0 ? -m.bl : 0;
    const int row_max = max(max(m.row_end, m.bl > 0 ? 2 : 0), m.el > 0 ? m.row_end + m.el - 1 : 0);
    CigarWalk cw;
    cw.start(A.op_len + m.op_off, A.op_chr + m.op_off, m.n_ops);
    int ring_lo[kRing], ring_hi[kRing];   // listed cells of path rows r-B .. r+B (lo > hi: none), slot = row mod ring
#pragma unroll
    for (int i = 0; i < kRing; i++) { ring_lo[i] = 1000000; ring_hi[i] = -1000000; }
    const int ring = 2 * B + 1;
    double ret = ninf;
    int plo = 1, phi = 0;   // previous DP row's range (empty)
    bool failed = false;
    for (int r = row_min - B; r <= row_max + B; r++) {
      {   // listed cells of row R = r + B enter the window (rows are produced in ascending order, each once)
        const int R = r + B;
        int lo = 1000000, hi = -1000000;
        if (R >= row_min && R <= row_max) {
          int a_, b_;
          if (R >= 0 && cw.row(R, a_, b_)) { lo = a_; hi = b_; }
          if (m.bl > 0 && R >= -m.bl && R < 3) { lo = min(lo, 0); hi = max(hi, m.bl - 1); }                      // graph.cc:2188-2192
          if (m.el > 0 && R >= m.row_end && R < m.row_end + m.el) { lo = min(lo, m.col_end - m.el); hi = max(hi, m.col_end); }   // 2204-2208
        }
        const int slot = ((R % ring) + ring) % ring;
        ring_lo[slot] = lo;
        ring_hi[slot] = hi;
      }
      int l = 1000000, h = -1000000;
      for (int i = 0; i < ring; i++)
        if (ring_lo[i] <= ring_hi[i]) { l = min(l, ring_lo[i] - B); h = max(h, ring_hi[i] + B); }
      if (l > h) { plo = 1; phi = 0; continue; }
      if (h - l + 1 > m.width) { failed = true; break; }
      const int p1 = r + m.posstart - 1;
      const bool row_ok = p1 >= 0 && p1 < m.s1_len;
      const unsigned char c1 = row_ok ? s1[p1] : 0;
      const double up_lp = c1 == '\n' ? ninf : A.log_mismatch;   // MatchProbability(s1[.], '-'), graph.h:555-563
      double left = ninf;   // value of (row, col - 1); at the row's first cell there is none
      bool have_left = false;
      for (int c = l; c <= h; c++) {
        double v = c == 0 ? 0.0 : ninf;   // column 0: probability 1, graph.cc:2240-2244
        if (c != 0 && c - 1 >= 0 && c - 1 < m.s2_len && row_ok) {
          const unsigned char c2 = s2[c - 1];
          if (c - 1 >= plo && c - 1 <= phi)
            v = lse_add(v, __dadd_rn(prev[c - 1 - plo], (c1 == '\n' || c2 == '\n') ? ninf : (c1 != c2 ? A.log_mismatch : A.log_match)));
          if (c >= plo && c <= phi) v = lse_add(v, __dadd_rn(prev[c - plo], up_lp));
          if (have_left) v = lse_add(v, __dadd_rn(left, c2 == '\n' ? ninf : A.log_mismatch));
          if (c == m.s2_len) ret = lse_add(ret, v);
        }
        cur[c - l] = v;
        left = v;
        have_left = true;
      }
      double* t = prev; prev = cur; cur = t;
      plo = l;
      phi = h;
    }
    if (failed) {
      atomicOr(A.error_flag, 1u);
      ret = NAN;
    }
    A.out[a] = ret;
  }
}

// ---- per-evaluation tables, reduction of partials -------------------------------------------
// comb_base[store] / comb_map[store]: paired sets keep a second copy of the first slot word in a table indexed by MATE 1's
// key id that holds, side by side, the word of that key in mate 1's store and the word of the same key (same node
// sequence) in mate 2's store (base + 1, index through the mate-2 -> mate-1 key map): tier 1 of the streaming kernel
// fetches both with one 256-bit gather for the pairs whose mates lie under the same key (nearly all of them).
// A patched full evaluation (engine.cu "patched full evaluation") applies the resident updates of the base walk list
// and, behind them, the few updates of the keys whose occurrences differ from the base's; the base entries of those keys
// (indices in the ascending list `skip`) are left out, so every key is written by exactly one thread and a key that lost
// its last occurrence simply keeps a stale epoch.
template <bool kInline>
__global__ void apply_slots_kernel(const SlotUpdate* upd, int n, const SlotUpdate* patch, int n_patch, const int32_t* skip, int n_skip,
                                   SlotA* const* tab_a, SlotB* const* tab_b, SlotA* const* comb_base,
                                   const int32_t* const* comb_map, const StoreTables T, uint32_t epoch, unsigned long long* flags,
                                   int n_flag_words, unsigned long long* timeline) {
  pdl_release();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  tl_begin(timeline, kTlApply);
  if (i < n_flag_words) flags[i] = 0ull;   // scratch cursor, error flag, overflow counters, tickets, accumulators
  if (i >= n + n_patch) {
    tl_end(timeline, kTlApply);
    return;
  }
  if (i < n && n_skip > 0) {
    int lo = 0, hi = n_skip;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (__ldg(skip + mid) < i) lo = mid + 1; else hi = mid;
    }
    if (lo < n_skip && __ldg(skip + lo) == i) {
      tl_end(timeline, kTlApply);
      return;
    }
  }
  const SlotUpdate u = i < n ? upd[i] : patch[i - n];
  SlotA a;
  a.epoch_flag = epoch | (u.n_occ > 1 ? 0x80000000u : 0u);
  a.walk = u.first.walk;
  a.cur_pos = u.first.cur_pos;
  a.skip_below = u.first.skip_below;
  SlotB b;
  b.seg = u.first.seg;
  b.n_occ = u.n_occ;
  b.occ_begin = u.occ_begin;
  b.pad = 0;
  (kInline ? T.a[u.store] : tab_a[u.store])[u.key] = a;
  (kInline ? T.b[u.store] : tab_b[u.store])[u.key] = b;
  SlotA* cb = kInline ? T.cb[u.store] : comb_base[u.store];
  if (cb) {
    const int32_t* mp = kInline ? T.cm[u.store] : comb_map[u.store];
    const int idx = mp ? mp[u.key] : u.key;
    if (idx >= 0) {   // 64-byte entry per mate-1 key: {first word mate 1, first word mate 2, second word mate 1, second word mate 2}
      cb[4 * idx] = a;
      SlotA bw;
      bw.epoch_flag = (uint32_t)b.seg;
      bw.walk = b.n_occ;
      bw.cur_pos = b.occ_begin;
      bw.skip_below = 0;
      cb[4 * idx + 2] = bw;
    }
  }
  tl_end(timeline, kTlApply);
}

// ---- CSR build: arena (key-major) -> rows (read-major) --------------------------------------
__global__ void count_reads_kernel(const int4* arena, size_t n, uint32_t* counts) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    atomicAdd(counts + arena[i].x, 1u);
}

template <bool kLong>
__global__ void fill_rows_kernel(const int4* arena, size_t n, const uint32_t* rowptr, uint32_t* cursor, int4* rows) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int4 a = arena[i];
    const uint32_t slot = rowptr[a.x] + atomicAdd(cursor + a.x, 1u);
    int4 r;
    if (kLong) { r.x = a.y; r.y = (int)(uint32_t)i; r.z = a.z; r.w = a.w; }   // {key, seq, logprob}
    else { r.x = a.w; r.y = a.y; r.z = a.z; r.w = (int)(uint32_t)i; }          // {key, pos, edor, seq}
    rows[slot] = r;
  }
}

// Atomics scatter in arbitrary order; restore arena (= reference list) order inside every read's row, then
// (short stores) publish the dense first-record array of the hybrid layout.
template <bool kLong>
__global__ void sort_rows_kernel(const uint32_t* rowptr, int n_reads, int4* rows, int4* first) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_reads) return;
  const uint32_t b = rowptr[r], e = rowptr[r + 1];
  for (uint32_t i = b + 1; i < e; i++) {
    const int4 v = rows[i];
    const uint32_t sv = kLong ? (uint32_t)v.y : (uint32_t)v.w;
    uint32_t j = i;
    while (j > b) {
      const int4 u = rows[j - 1];
      const uint32_t su = kLong ? (uint32_t)u.y : (uint32_t)u.w;
      if (su <= sv) break;
      rows[j] = u;
      j--;
    }
    rows[j] = v;
  }
  if (!kLong) {
    int4 f;
    if (e > b) {
      f = rows[b];
      const uint32_t cnt = e - b;
      f.z |= (int)((cnt < 0x3fffu ? cnt : 0x3fffu) << 16);
      f.w = (int)b;
    } else {
      f.x = -1; f.y = 0; f.z = 0; f.w = 0;
    }
    first[r] = f;
  }
}

// Static tier-2 list: reads owning more than one record on some mate, in read-id order (scan, not atomics,
// so the list — and with it the association of the partial sums — is the same on every run).
// class of a read for the static list: 0 = tier 1 (at most one record per mate), else 1 + rank, where the shapes
// tier 2 streams come first — (1,2) (2,1) (2,2) (0,2) (2,0) = ranks 0..4 — and the shapes with three or more records
// on a mate (the multi pass's static part) after them.
__device__ __forceinline__ int complex_class(const int4* first1, const int4* first2, int r) {
  const int c1 = (first1[r].z >> 16) & 0x3fff;
  const int c2 = first2 ? ((first2[r].z >> 16) & 0x3fff) : 0;
  if (c1 < 2 && c2 < 2) return 0;
  const int id = min(c1, 3) * 4 + min(c2, 3);
  //                       id: 0   1   2  3   4   5   6  7  8  9  10 11 12 13 14  15
  constexpr int kRank[16] = {12, 13, 3, 5, 14, 15, 0, 6, 4, 1, 2, 7, 8, 9, 10, 11};
  return 1 + kRank[id];
}

__global__ void complex_flags_kernel(const int4* first1, const int4* first2, int n_reads, uint32_t* flags, int cls) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r > n_reads) return;
  flags[r] = (r < n_reads && complex_class(first1, first2, r) == cls) ? 1u : 0u;
}

__global__ void complex_scatter_kernel(const int4* first1, const int4* first2, int n_reads, const uint32_t* offs,
                                       uint32_t* list, int cls) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_reads) return;
  if (complex_class(first1, first2, r) == cls) list[offs[r]] = (uint32_t)r;
}

__global__ void compact_count_kernel(const uint32_t* list, int n_complex, const uint32_t* rowptr, uint32_t* cptr,
                                     const uint32_t* lens, uint32_t* clens) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k > n_complex) return;
  uint32_t c = 0;
  if (k < n_complex) {
    const uint32_t r = list[k];
    c = rowptr[r + 1] - rowptr[r];
    if (clens) clens[k] = lens[r];
  }
  cptr[k] = c;
}

__global__ void cdesc_fill_kernel(const uint32_t* list, int n_complex, const uint32_t* lens, const uint32_t* cptr1,
                                  const uint32_t* cptr2, int4* desc) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_complex) return;
  const uint32_t r = list[k];
  desc[k] = make_int4((int)r, (int)lens[r], (int)cptr1[k], cptr2 ? (int)cptr2[k] : 0);
}

__global__ void compact_copy_kernel(const uint32_t* list, int n_complex, const uint32_t* rowptr, const uint32_t* cptr,
                                    const int4* rows, int4* crows) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_complex) return;
  const uint32_t r = list[k];
  const uint32_t b = rowptr[r], n = rowptr[r + 1] - b, d = cptr[k];
  for (uint32_t i = 0; i < n; i++) crows[d + i] = rows[b + i];
}

// ---- cache append: new records of reads that are scored already -------------------------------------------------------
// A key inserted after the device index was built (the annealing loop aligns a new join's window on demand, graph.cc:
// 1967-1968) brings a few hundred records. Instead of rebuilding the read-major index over all records, each read that
// gains records gets its row block RELOCATED to the tail of the row array with the new rows appended (they are the
// highest arena indices, i.e. last in reference list order), its first-record word is updated, and the read is flagged:
// in `dirty`, and in its packed / fast pair record ("elsewhere") so that the list-driven phases leave it to the appendix
// phase. One thread per affected read; the host supplies exact destinations (it keeps every read's record count).
struct AppendGroup { uint32_t read; uint32_t new_begin; uint32_t n_new; uint32_t dst; };   // dst: new row block's first row
// The whole of one cache append in ONE launch over one staged blob: both mates' new arena records to the arena tails,
// both mates' relocated row blocks, the newly flagged reads onto the appendix list, the key-map entries that changed.
// One thread per item of the concatenated index space; the parts touch disjoint memory.
__global__ void append_apply_kernel(const AppendJob J) {
  const uint32_t n_a0 = J.m[0].n_rec, n_a1 = J.m[1].n_rec, n_g0 = (uint32_t)J.m[0].n_groups, n_g1 = (uint32_t)J.m[1].n_groups;
  const uint32_t total = n_a0 + n_a1 + n_g0 + n_g1 + (uint32_t)J.n_appx_new + (uint32_t)J.n_p12 + (uint32_t)J.n_p21;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    uint32_t k = i;
    if (k < n_a0) { static_cast<int4*>(J.m[0].arena_dst)[k] = static_cast<const int4*>(J.m[0].arena_src)[k]; continue; }
    k -= n_a0;
    if (k < n_a1) { static_cast<int4*>(J.m[1].arena_dst)[k] = static_cast<const int4*>(J.m[1].arena_src)[k]; continue; }
    k -= n_a1;
    if (k < n_g0 + n_g1) {
      const int m = k < n_g0 ? 0 : 1;
      if (m) k -= n_g0;
      const AppendGroup ag = static_cast<const AppendGroup*>(J.m[m].groups)[k];
      const int4* new_rows = static_cast<const int4*>(J.m[m].new_rows);
      int4* rows = static_cast<int4*>(J.m[m].rows);
      int4* first = static_cast<int4*>(J.m[m].first);
      int4 f = first[ag.read];
      const uint32_t cnt_old = f.x < 0 ? 0u : (uint32_t)((f.z >> 16) & 0x3fff);
      const uint32_t base_old = (uint32_t)f.w;
      for (uint32_t t = 0; t < cnt_old; t++) rows[ag.dst + t] = rows[base_old + t];
      for (uint32_t t = 0; t < ag.n_new; t++) rows[ag.dst + cnt_old + t] = new_rows[ag.new_begin + t];
      if (cnt_old == 0) {
        const int4 r0 = new_rows[ag.new_begin];   // {key, pos, edor, seq}
        f.x = r0.x;
        f.y = r0.y;
        f.z = r0.z & 0x4000ffff;
      }
      f.z = (f.z & 0x4000ffff) | (int)((cnt_old + ag.n_new) << 16);
      f.w = (int)ag.dst;
      first[ag.read] = f;
      J.dirty[ag.read] = 1u;
      // (a read that gained records on both mates is flagged by two threads: both write the same bit)
      if (J.pairs) atomicOr(&static_cast<uint4*>(J.pairs)[ag.read].x, 0x80000000u);   // PackedPair: "tier 2" = not tier 1's
      if (J.fast) atomicOr(&static_cast<uint4*>(J.fast)[ag.read].x, 0x80000000u);     // FastPair: "elsewhere"
      continue;
    }
    k -= n_g0 + n_g1;
    if (k < (uint32_t)J.n_appx_new) { J.appx_dst[k] = J.appx_src[k]; continue; }
    k -= (uint32_t)J.n_appx_new;
    if (k < (uint32_t)J.n_p12) { const int2 p = J.p12_patch[k]; J.p12[p.x] = p.y; continue; }
    k -= (uint32_t)J.n_p12;
    const int2 p = J.p21_patch[k];
    J.p21[p.x] = p.y;
  }
}
// per-read record counts of a store after a full build (the host keeps them up to date across appends)
__global__ void extract_counts_kernel(const int4* first, const uint32_t* rowptr, int n, uint16_t* out) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const uint32_t c = rowptr[r + 1] - rowptr[r];
  out[r] = (uint16_t)(c < 0xffffu ? c : 0xffffu);
  (void)first;
}
int grid_for(size_t n, int block, int sm_count, int per_sm) {
  size_t need = (n + block - 1) / block;
  size_t cap = (size_t)sm_count * per_sm;
  return (int)(need < 1 ? 1 : (need < cap ? need : cap));
}

}  // namespace

void launch_append_apply(const AppendJob& J, cudaStream_t st) {
  const size_t total = (size_t)J.m[0].n_rec + J.m[1].n_rec + (size_t)J.m[0].n_groups + (size_t)J.m[1].n_groups + (size_t)J.n_appx_new +
                       (size_t)J.n_p12 + (size_t)J.n_p21;
  if (total == 0) return;
  const size_t blocks = (total + 127) / 128;
  append_apply_kernel<<<(unsigned)(blocks < 1184 ? blocks : 1184), 128, 0, st>>>(J);
}
void launch_extract_counts(const void* first, const uint32_t* rowptr, int n, uint16_t* out, cudaStream_t st) {
  if (n > 0) extract_counts_kernel<<<(n + 255) / 256, 256, 0, st>>>(static_cast<const int4*>(first), rowptr, n, out);
}

// ---- launch wrappers ------------------------------------------------------------------------
// Grids are sized to exactly one resident wave (SM count x blocks that fit per SM for that kernel) so the
// grid-stride loops have no partial second wave.
// The streaming kernel's instantiation: penalised sets (coverage events) and sets whose records do not fit PackedPair
// stream the 16-byte first records; everything else the packed pairs.
using StreamKernel = void (*)(const ScoreParams);
// The streaming kernel's instantiation. Penalised sets (coverage events) and sets whose records do not fit PackedPair
// stream the 16-byte first records; sets of uniform read length with a term table take the tabulated body. The
// (resident blocks, reads per lane) shape of the tabulated body can be overridden for measurements with
// GAML_B200_STREAM_SHAPE=<blocks><reads>, e.g. 62 = 6 blocks per SM, two reads per lane.
StreamKernel stream_kernel(bool cov, bool packed, bool tab) {
  if (cov) return paired_stream_kernel<true, false, false, 4, 2>;
  if (!packed) return paired_stream_kernel<false, false, false, 4, 2>;
  if (!tab) return paired_stream_kernel<false, true, false, 4, 2>;
  const char* env = getenv("GAML_B200_STREAM_SHAPE");   // (read per launch: a measurement script switches shapes in one process)
  switch (env ? atoi(env) : 0) {
    case 42: return paired_stream_kernel<false, true, true, 4, 2>;
    case 52: return paired_stream_kernel<false, true, true, 5, 2>;
    case 44: return paired_stream_kernel<false, true, true, 4, 4>;
    case 32: return paired_stream_kernel<false, true, true, 3, 2>;
    case 2: return nullptr;   // two launches: stream_kernel_tier1 + stream_kernel_rest
    // measured (profiles/r02_summary.md): one fused launch at 4 blocks x 2 reads beats every two-launch shape — tier 1 is
    // bound by DRAM, and MORE resident warps make it slower, not faster
    default: return paired_stream_kernel<false, true, true, 4, 2>;
  }
}
// The two-launch form of a set with fast records: tier 1 alone (shape from GAML_B200_TIER1_SHAPE=<blocks><reads>), then the rest.
StreamKernel stream_kernel_tier1() {
  const char* env = getenv("GAML_B200_TIER1_SHAPE");
  switch (env ? atoi(env) : 0) {
    case 81: return paired_stream_kernel<false, true, true, 8, 1, 1>;
    case 61: return paired_stream_kernel<false, true, true, 6, 1, 1>;
    case 62: return paired_stream_kernel<false, true, true, 6, 2, 1>;
    case 52: return paired_stream_kernel<false, true, true, 5, 2, 1>;
    case 42: return paired_stream_kernel<false, true, true, 4, 2, 1>;
    case 44: return paired_stream_kernel<false, true, true, 4, 4, 1>;
    case 34: return paired_stream_kernel<false, true, true, 3, 4, 1>;
    case 82: return paired_stream_kernel<false, true, true, 8, 2, 1>;
    default: return paired_stream_kernel<false, true, true, 6, 2, 1>;
  }
}
StreamKernel stream_kernel_rest() { return paired_stream_kernel<false, true, true, 4, 2, 2>; }

template <class K>
int resident_blocks(K kernel, int block) {
  int n = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, block, 0) != cudaSuccess || n < 1) n = 1;
  return n;
}

int score_grid(int which, int n_items, int sm_count) {
  static int per_sm[6] = {0, 0, 0, 0, 0, 0};
  if (which < 0 || which > 5) which = 0;
  if (per_sm[which] == 0) {
    switch (which) {
      case kGridPairedFull: per_sm[which] = resident_blocks(stream_kernel(false, true, false), kBlock); break;
      case kGridPairedComplex: per_sm[which] = resident_blocks(stream_kernel(false, true, false), kBlock); break;
      case kGridPairedTotal: per_sm[which] = resident_blocks(paired_total_kernel, kBlock); break;
      case kGridSingleFull: per_sm[which] = resident_blocks(single_full_kernel, kBlock); break;
      case kGridSingleComplex: per_sm[which] = resident_blocks(single_complex_kernel, kBlock); break;
      default: per_sm[which] = resident_blocks(pacbio_full_kernel, kBlock); break;
    }
  }
  return grid_for((size_t)n_items, kBlock, sm_count, per_sm[which]);
}
// The many-placement passes' list length is unknown at launch: one block per SM, grid-stride beyond (they usually find
// nothing, or a few hundred reads; every extra block is an extra trip through the tail of the chain).
int overflow_grid(int sm_count) { return sm_count; }

// One kernel of an evaluation's chain; pdl = launched as a programmatic dependent of the kernel before it on `st`.
thread_local LaunchList* g_recorder = nullptr;
void set_launch_recorder(LaunchList* list) { g_recorder = list; }

cudaError_t issue_launch(const PendingLaunch& pl, cudaStream_t st) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(pl.grid);
  cfg.blockDim = dim3(pl.block);
  cfg.stream = st;
  cudaLaunchAttribute attr{};
  attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr.val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = &attr;
  cfg.numAttrs = pl.pdl ? 1 : 0;
  return cudaLaunchKernelExC(&cfg, pl.func, const_cast<void**>(pl.arg_ptrs));
}

template <class T>
void pack_arg(PendingLaunch& pl, size_t& off, const T& v) {
  off = (off + alignof(T) - 1) & ~(alignof(T) - 1);
  memcpy(pl.arg_buf + off, &v, sizeof(T));
  pl.arg_ptrs[pl.n_args++] = pl.arg_buf + off;
  off += sizeof(T);
}

template <class... KArgs, class... Args>
void launch_chain(void (*kernel)(KArgs...), int grid, int block, cudaStream_t st, bool pdl, Args&&... args) {
  static_assert(sizeof...(KArgs) == sizeof...(Args), "argument count");
  static_assert(sizeof...(KArgs) <= sizeof(PendingLaunch::arg_ptrs) / sizeof(void*), "too many kernel arguments");
  static_assert((sizeof(KArgs) + ... + 0) + 16 * sizeof...(KArgs) <= sizeof(PendingLaunch::arg_buf), "argument buffer too small");
  PendingLaunch local;
  LaunchList* rec = g_recorder;
  PendingLaunch& pl = (rec && rec->n < 16) ? rec->item[rec->n] : local;
  pl.func = reinterpret_cast<const void*>(kernel);
  pl.grid = (unsigned)grid;
  pl.block = (unsigned)block;
  pl.pdl = pdl;
  pl.n_args = 0;
  size_t off = 0;
  (pack_arg<std::remove_cv_t<std::remove_reference_t<KArgs>>>(pl, off, static_cast<std::remove_cv_t<std::remove_reference_t<KArgs>>>(args)), ...);
  if (rec && rec->n < 16) {
    rec->n++;
    return;
  }
  issue_launch(pl, st);
}

void launch_apply_slots(const SlotUpdate* upd, int n, const SlotUpdate* patch, int n_patch, const int32_t* skip, int n_skip,
                        SlotA* const* tab_a, SlotB* const* tab_b, SlotA* const* comb_base,
                        const int32_t* const* comb_map, const StoreTables* inline_tabs, uint32_t epoch, unsigned long long* flags,
                        int n_flag_words, unsigned long long* timeline, cudaStream_t st) {
  const int m = n + n_patch > n_flag_words ? n + n_patch : n_flag_words;
  if (inline_tabs)
    launch_chain(apply_slots_kernel<true>, (m + 255) / 256, 256, st, false, upd, n, patch, n_patch, skip, n_skip, tab_a, tab_b, comb_base,
                 comb_map, *inline_tabs, epoch, flags, n_flag_words, timeline);
  else
    launch_chain(apply_slots_kernel<false>, (m + 255) / 256, 256, st, false, upd, n, patch, n_patch, skip, n_skip, tab_a, tab_b, comb_base,
                 comb_map, StoreTables{}, epoch, flags, n_flag_words, timeline);
}

// Every wrapper below appends its kernels to the evaluation's chain. `chained` = the operation before it on `st` is a
// kernel of the chain (so the first kernel may be a programmatic dependent too). With `profile` the streaming
// kernel(s) of the set are bracketed by e0/e1 (the roofline timing); an event between two kernels makes the second
// wait for the first in the ordinary way, so profiling costs the overlap at those two boundaries.
// Tier 1 and tier 2 touch disjoint reads and only meet in the (commutative, integer) accumulators.
int launch_paired_full(const ScoreParams& P, int grid, int cgrid, uint32_t n_multi_items, int ovf_grid, int sm_count,
                       cudaStream_t st, bool chained, bool profile, cudaEvent_t e0, cudaEvent_t e1, bool tail) {
  int n_launched = 0;
  // chain: [multi pass] -> streaming kernel (tier 1 + tier 2) [-> many-placement pass]. Without the trailing pass (!tail)
  // the streaming kernel ends the chain: it publishes the final line when it listed no read, else a pending one, and
  // the owning host runs the pass on demand (launch_paired_tail). The trailing pass would otherwise wait with 148
  // register-hungry blocks that cannot become resident before streaming blocks retire. Only two kernels of a chain are in
  // flight at a time (kernel n+2 starts when kernel n has completed), so the multi pass — a small grid of
  // register-hungry blocks with a long dependent chain, needing apply_slots only — goes FIRST and runs underneath the
  // streaming kernel, whose tile counters absorb the register file it holds meanwhile. It waits for apply_slots at its
  // top and releases after; the streaming kernel then starts without waiting and waits at its END, which makes
  // completion transitive for the last kernel. (cgrid is unused here: tier 2 is a phase of the streaming kernel.)
  (void)cgrid;
  tail = tail || profile;
  ScoreParams Q = P;
  bool dep = chained && !profile;
  bool first = true;
  if (n_multi_items > 0 || P.n_appx > 0) {
    Q.chain_first = 1;
    Q.finish_here = 0;
    if (n_multi_items < (uint32_t)P.n_appx) n_multi_items = (uint32_t)P.n_appx;   // (grid sizing only)
    // at most ONE resident wave: the streaming kernel behind it is released only when every block of this grid has
    // started, so blocks queuing for a second wave would hold it back for the duration of the first
    static const int per_sm = resident_blocks(paired_multi_kernel, kOvfBlock);
    launch_chain(paired_multi_kernel, grid_for(n_multi_items, kOvfBlock, sm_count, per_sm), kOvfBlock, st, dep, Q);
    n_launched++;
    dep = true;
    first = false;
  }
  if (profile) cudaEventRecord(e0, st);
  Q.chain_first = first || profile ? 1 : 0;
  Q.finish_here = profile ? 0 : (tail ? 1 : 2);   // when profiling, e0/e1 bracket the streaming work alone: the last kernel publishes
  {
    // one resident wave of the instantiation that runs (its blocks draw tiles from counters)
    static StreamKernel seen[16];
    static int seen_per_sm[16];
    static int n_seen = 0;
    auto blocks_per_sm = [&](StreamKernel k) {
      for (int i = 0; i < n_seen; i++)
        if (seen[i] == k) return seen_per_sm[i];
      const int v = resident_blocks(k, kBlock);
      if (n_seen < 16) { seen[n_seen] = k; seen_per_sm[n_seen++] = v; }
      return v;
    };
    const bool tab = P.pairs != nullptr && P.comb != nullptr && P.fast != nullptr;
    const StreamKernel k = stream_kernel(P.ev_keys != nullptr, P.pairs != nullptr, tab);
    if (k) {
      grid = grid_for((size_t)P.n_reads, kBlock, sm_count, blocks_per_sm(k));
      launch_chain(k, grid, kBlock, st, dep && !profile, Q);
      n_launched++;
    } else {
      // fast records: tier 1 in a launch of its own, everything else in the next one (which waits for it at its end)
      ScoreParams Q1 = Q;
      Q1.finish_here = 0;
      const StreamKernel k1 = stream_kernel_tier1(), k2 = stream_kernel_rest();
      launch_chain(k1, grid_for((size_t)std::max(P.n_tier1, 1), kBlock, sm_count, blocks_per_sm(k1)), kBlock, st, dep && !profile, Q1);
      ScoreParams Q2 = Q;
      Q2.chain_first = 0;
      const int items = std::max(std::max(P.n_main, P.n_complex - P.n_main), std::max(P.n_cross / 2, P.n_appx));
      launch_chain(k2, grid_for((size_t)std::max(items, 1), kBlock, sm_count, blocks_per_sm(k2)), kBlock, st, true, Q2);
      n_launched += 2;
    }
  }
  if (profile) cudaEventRecord(e1, st);
  if (!tail) return n_launched;
  launch_chain(paired_overflow_kernel, ovf_grid, kOvfBlock, st, !profile, P, 1);
  return n_launched + 1;
}

void launch_paired_tail(const ScoreParams& P, int ovf_grid, cudaStream_t st) {
  launch_chain(paired_overflow_kernel, ovf_grid, kOvfBlock, st, false, P, 1);
}

void launch_paired_delta(const ScoreParams& P, uint32_t n_touch_records, int grid_total, int ovf_grid, int sm_count,
                         cudaStream_t st, bool chained, bool profile, cudaEvent_t e0, cudaEvent_t e1) {
  if (profile) cudaEventRecord(e0, st);
  bool dep = chained && !profile;
  if (n_touch_records > 0) {
    static const int per_sm = resident_blocks(paired_delta_kernel, kOvfBlock);   // one resident wave, grid-stride beyond
    launch_chain(paired_delta_kernel, grid_for(n_touch_records, kOvfBlock, sm_count, per_sm), kOvfBlock, st, dep, P);
    dep = true;
  }
  if (P.delta_only) {
    // total length unchanged since the running total was formed: the touched reads' terms were swapped in place, the
    // many-placement pass finishes the set (it runs even with nothing to do: it publishes the result)
    launch_chain(paired_overflow_kernel, n_touch_records > 0 ? ovf_grid : 1, kOvfBlock, st, dep, P, 2);
  } else {
    if (n_touch_records > 0) launch_chain(paired_overflow_kernel, ovf_grid, kOvfBlock, st, true, P, 0);
    launch_chain(paired_total_kernel, grid_total, kBlock, st, dep, P);
  }
  if (profile) cudaEventRecord(e1, st);
}

void launch_single_full(const ScoreParams& P, int grid, int cgrid, int ovf_grid, cudaStream_t st, bool chained, bool profile,
                        cudaEvent_t e0, cudaEvent_t e1) {
  if (profile) cudaEventRecord(e0, st);
  launch_chain(single_full_kernel, grid, kBlock, st, chained && !profile, P);
  if (cgrid > 0) launch_chain(single_complex_kernel, cgrid, kBlock, st, true, P);
  if (profile) cudaEventRecord(e1, st);
  launch_chain(single_overflow_kernel, ovf_grid, kOvfBlock, st, !profile, P);
}

void launch_pacbio_full(const ScoreParams& P, int grid, int ovf_grid, cudaStream_t st, bool chained, bool profile, cudaEvent_t e0,
                        cudaEvent_t e1) {
  if (profile) cudaEventRecord(e0, st);
  launch_chain(pacbio_full_kernel, grid, kBlock, st, chained && !profile, P);
  if (profile) cudaEventRecord(e1, st);
  launch_chain(pacbio_overflow_kernel, ovf_grid, kOvfBlock, st, !profile, P);
}

cudaError_t build_csr(const void* arena, size_t n_records, int n_reads, bool is_long, uint32_t* rowptr, uint32_t* cursor,
                      void* rows, void* first, void* temp, size_t temp_bytes, int sm_count, cudaStream_t st, int* launches) {
  // rowptr doubles as the count array (n_reads + 1 entries, zeroed here)
  cudaError_t err = cudaMemsetAsync(rowptr, 0, sizeof(uint32_t) * ((size_t)n_reads + 1), st);
  if (err != cudaSuccess) return err;
  err = cudaMemsetAsync(cursor, 0, sizeof(uint32_t) * ((size_t)n_reads + 1), st);
  if (err != cudaSuccess) return err;
  if (n_records > 0) {
    count_reads_kernel<<<grid_for(n_records, 256, sm_count, 16), 256, 0, st>>>(static_cast<const int4*>(arena), n_records, rowptr);
    (*launches)++;
  }
  size_t need = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, need, rowptr, rowptr, n_reads + 1, st);
  if (need > temp_bytes) return cudaErrorMemoryAllocation;
  err = cub::DeviceScan::ExclusiveSum(temp, need, rowptr, rowptr, n_reads + 1, st);
  if (err != cudaSuccess) return err;
  (*launches)++;
  if (n_records > 0) {
    const int g = grid_for(n_records, 256, sm_count, 16);
    if (is_long) fill_rows_kernel<true><<<g, 256, 0, st>>>(static_cast<const int4*>(arena), n_records, rowptr, cursor, static_cast<int4*>(rows));
    else fill_rows_kernel<false><<<g, 256, 0, st>>>(static_cast<const int4*>(arena), n_records, rowptr, cursor, static_cast<int4*>(rows));
    (*launches)++;
  }
  if (n_reads > 0) {
    const int gs = (n_reads + 255) / 256;
    if (is_long) sort_rows_kernel<true><<<gs, 256, 0, st>>>(rowptr, n_reads, static_cast<int4*>(rows), nullptr);
    else sort_rows_kernel<false><<<gs, 256, 0, st>>>(rowptr, n_reads, static_cast<int4*>(rows), static_cast<int4*>(first));
    (*launches)++;
  }
  return cudaGetLastError();
}

// Builds the static tier-2 list; flags must hold n_reads + 1 uint32 (scratch), list n_reads uint32. The number
// of listed reads is left in flags[n_reads] (exclusive scan total).
cudaError_t build_complex_list(const void* first1, const void* first2, int n_reads, uint32_t* flags, uint32_t* list,
                               void* temp, size_t temp_bytes, cudaStream_t st, int* launches, uint32_t* n_complex_out,
                               int32_t* class_begin /* 17 */) {
  // The list is ordered by (record-count class, read id): warps of the tier-2 kernel then hold reads of one shape
  // — (2,1), (1,2), (2,2), ... — and do not execute each other's paths. One flag/scan/scatter pass per class.
  const int g = (n_reads + 1 + 255) / 256;
  const int4* f1 = static_cast<const int4*>(first1);
  const int4* f2 = static_cast<const int4*>(first2);
  size_t need = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, need, flags, flags, n_reads + 1, st);
  if (need > temp_bytes) return cudaErrorMemoryAllocation;
  uint32_t base = 0;
  class_begin[0] = 0;
  for (int cls = 1; cls <= 16; cls++) {
    class_begin[cls - 1] = (int32_t)base;   // kernel-side class id = cls - 1 = min(cnt1,3)*4 + min(cnt2,3)
    complex_flags_kernel<<<g, 256, 0, st>>>(f1, f2, n_reads, flags, cls);
    cudaError_t err = cub::DeviceScan::ExclusiveSum(temp, need, flags, flags, n_reads + 1, st);
    if (err != cudaSuccess) return err;
    uint32_t cnt = 0;
    err = cudaMemcpyAsync(&cnt, flags + n_reads, 4, cudaMemcpyDeviceToHost, st);
    if (err != cudaSuccess) return err;
    err = cudaStreamSynchronize(st);
    if (err != cudaSuccess) return err;
    (*launches) += 2;
    if (cnt > 0) {
      complex_scatter_kernel<<<(n_reads + 255) / 256, 256, 0, st>>>(f1, f2, n_reads, flags, list + base, cls);
      (*launches)++;
      base += cnt;
    }
  }
  class_begin[16] = (int32_t)base;
  *n_complex_out = base;
  return cudaGetLastError();
}

// Compact tier-2 store of one mate, step 1: per-list-entry record counts -> exclusive scan into cptr (n_complex+1
// entries; the total is left in cptr[n_complex]); clens (optional) receives the packed lengths of the listed reads.
cudaError_t compact_offsets(const uint32_t* list, int n_complex, const uint32_t* rowptr, uint32_t* cptr, const uint32_t* lens,
                            uint32_t* clens, void* temp, size_t temp_bytes, cudaStream_t st, int* launches) {
  compact_count_kernel<<<(n_complex + 1 + 255) / 256, 256, 0, st>>>(list, n_complex, rowptr, cptr, lens, clens);
  size_t need = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, need, cptr, cptr, n_complex + 1, st);
  if (need > temp_bytes) return cudaErrorMemoryAllocation;
  cudaError_t err = cub::DeviceScan::ExclusiveSum(temp, need, cptr, cptr, n_complex + 1, st);
  (*launches) += 2;
  return err != cudaSuccess ? err : cudaGetLastError();
}

// step 2: copy the listed reads' rows (already in reference list order) next to each other.
cudaError_t compact_copy(const uint32_t* list, int n_complex, const uint32_t* rowptr, const uint32_t* cptr, const void* rows,
                         void* crows, cudaStream_t st, int* launches) {
  if (n_complex > 0) {
    compact_copy_kernel<<<(n_complex + 255) / 256, 256, 0, st>>>(list, n_complex, rowptr, cptr, static_cast<const int4*>(rows),
                                                               static_cast<int4*>(crows));
    (*launches)++;
  }
  return cudaGetLastError();
}

void launch_batch(const ScoreParams& P, const BatchParams& B, uint32_t n_touch_records, double* out, const uint32_t* error_flag,
                  int sm_count, cudaStream_t st) {
  // GAML_B200_BATCH_TIMING=1 (measurement aid): per-kernel device times of the batch on stderr
  static const bool timing = getenv("GAML_B200_BATCH_TIMING") != nullptr;
  cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
  if (timing)
    for (auto& e : ev) cudaEventCreate(&e);
  if (timing) cudaEventRecord(ev[0], st);
  // base pass: chunks of at most kBatchMaxLen distinct lengths, each with its own nb + 1 bins
  const int gx = grid_for((size_t)P.n_reads, kBlock, sm_count, 4);
  int chunk = 0;
  for (int j0 = 0; j0 < B.n_len; j0 += kBatchMaxLen, chunk++) {
    const int nb = B.n_len - j0 < kBatchMaxLen ? B.n_len - j0 : kBatchMaxLen;
    batch_base_kernel<<<gx, kBlock, 0, st>>>(P, B, j0, nb, (size_t)chunk * (kBatchMaxLen + 1));
  }
  if (timing) cudaEventRecord(ev[1], st);
  chunk = 0;
  for (int j0 = 0; j0 < B.n_len; j0 += kBatchMaxLen, chunk++) {
    const int nb = B.n_len - j0 < kBatchMaxLen ? B.n_len - j0 : kBatchMaxLen;
    batch_prefix_kernel<<<1, kBatchMaxLen, 0, st>>>(B, j0, nb, (size_t)chunk * (kBatchMaxLen + 1));
  }
  if (timing) cudaEventRecord(ev[2], st);
  if (n_touch_records > 0 && B.n_blocks > 0) batch_touch_kernel<<<B.n_blocks, kBlock, 0, st>>>(P, B);   // a block per slice of a candidate's records
  if (timing) cudaEventRecord(ev[3], st);
  batch_finalize_kernel<<<(B.n_cand + 127) / 128, 128, 0, st>>>(B, out, error_flag, (long long)P.n_reads);
  if (timing) {
    cudaEventRecord(ev[4], st);
    cudaEventSynchronize(ev[4]);
    float t[4];
    for (int i = 0; i < 4; i++) cudaEventElapsedTime(&t[i], ev[i], ev[i + 1]);
    fprintf(stderr, "[gaml_b200 batch] n_len %d: base %.3f ms, prefix %.3f ms, touch %.3f ms (%u records), finalize %.3f ms\n", B.n_len, t[0], t[1],
            t[2], n_touch_records, t[3]);
    for (auto& e : ev) cudaEventDestroy(e);
  }
}
int batch_hist_bins(int n_len) { return ((n_len + kBatchMaxLen - 1) / kBatchMaxLen) * (kBatchMaxLen + 1); }
int batch_launches(int n_len, bool touch) { return 2 * ((n_len + kBatchMaxLen - 1) / kBatchMaxLen) + (touch ? 1 : 0) + 1; }

// Term table of a paired set whose pairs all have the same read lengths: entry (e1, e2, d) = the pair term
// (p1*p2)*ins(d) (graph.cc:1859-1863, 1889, same order of products) and its fixed-point logarithm, by the very functions
// the kernels use on the fly, so a tabulated term and a recomputed one are the same bits.
__global__ void build_term_table_kernel(const double* p1, const double* p2, const double* ins, int ins_n, int shift, const double2* log_tab,
                                        TermEntry* out) {
  const size_t total = ((size_t)1 << (2 * shift)) * (size_t)ins_n;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int d = (int)(i % (size_t)ins_n);
    const int ee = (int)(i / (size_t)ins_n);
    const int e1 = ee >> shift, e2 = ee & ((1 << shift) - 1);
    const double t = __dmul_rn(__dmul_rn(p1[e1], p2[e2]), ins[d]);
    out[i + 1] = TermEntry{t, fix_log(log_tab, t)};
    if (i == 0) out[0] = TermEntry{0.0, kTermOdd};   // entry 0: "no pair term" (FastPair::w of a pair whose static filters fail)
  }
}
void launch_build_term_table(const double* p1, const double* p2, const double* ins, int ins_n, int shift, const void* log_tab, void* out,
                             int sm_count, cudaStream_t st) {
  const size_t total = ((size_t)1 << (2 * shift)) * (size_t)ins_n;
  build_term_table_kernel<<<grid_for(total, 256, sm_count, 8), 256, 0, st>>>(p1, p2, ins, ins_n, shift, static_cast<const double2*>(log_tab),
                                                                           static_cast<TermEntry*>(out));
}

// FastPair (16 B per pair, sets with a term table): what tier 1 needs of a pair whose mates both own exactly one record
// under the SAME key. Both records then share the key's offset in whatever walk holds it, so everything about the pair
// term except "is the key live, and do both records pass the skip rule" is a property of the two records — orientation
// / order filter, insert distance, (p1*p2)*ins and its logarithm — and is resolved here, once per cache commit, into an
// index into the term table:  x = key | noterm << 30 | elsewhere << 31,  y = pos1,  z = pos2,  w = term-table index
// (0 = the filters drop the pair: a term of +0.0). noterm: a mate without any record. elsewhere: the read is scored by
// another phase — tier 2 / rare shapes (several records on a mate) or the cross list (mates under different keys, or an
// edit distance beyond the table: the general body, tier1_body), for which flags[r] = 1 is emitted.
__global__ void pack_fast_kernel(const uint4* pairs, int n, int shift, int ins_n, uint32_t uniform_ll, uint4* out, uint32_t* flags) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r > n) return;
  if (r == n) { flags[r] = 0u; return; }
  const uint4 pr = pairs[r];
  const uint32_t key1 = pr.x & kPackKeyMask;
  const int e1 = (int)((pr.x >> kPackKeyBits) & kPackEdMask), e2 = (int)((pr.y >> kPackKeyBits) & kPackEdMask);
  const int xo = (int)((pr.x >> 29) & 1u), yo = (int)((pr.y >> 29) & 1u);
  const bool none = ((pr.x >> 30) & 1u) != 0u || ((pr.y >> 30) & 1u) != 0u;
  const bool tier2 = (pr.x >> 31) != 0u, same = (pr.y >> 31) != 0u;
  const int pos1 = (int)pr.z, pos2 = (int)pr.w;
  const int l1 = (int)(uniform_ll & 0xffff), l2 = (int)(uniform_ll >> 16);
  const bool fit = e1 < (1 << shift) && e2 < (1 << shift);
  uint4 v = make_uint4(0u, 0u, 0u, 0u);
  uint32_t cross = 0u;
  // the term-table index of (first record of mate 1, first record of mate 2) when both lie under one key: the pair term
  // of a fast read; for the others only a locality hint for the internal order (reads of like keys and terms together)
  uint32_t tix = 0u;
  if (!none && same && fit) {
    const bool fwd = pos1 < pos2;
    const int d = fwd ? pos2 - pos1 + l2 : pos1 - pos2 + l1;   // graph.cc:1866-1875 (both positions move by the same offset)
    const bool term = xo != yo && xo == (fwd ? 0 : 1) && (unsigned)d < (unsigned)ins_n;
    tix = term ? 1u + (uint32_t)((e1 << shift) | e2) * (uint32_t)ins_n + (uint32_t)d : 0u;
  }
  if (tier2) {
    v.x = 0x80000000u | key1;
    v.w = tix;
  } else if (none) {
    v.x = 0x40000000u;
  } else if (!same || !fit) {
    v.x = 0x80000000u | key1;
    cross = 1u;
  } else {
    v.x = key1;
    v.y = (uint32_t)pos1;
    v.z = (uint32_t)pos2;
    v.w = tix;
  }
  out[r] = v;
  flags[r] = cross;
}
// ---- internal read order ------------------------------------------------------------------------------------------
// Reads are scored in an INTERNAL order fixed at the first cache commit: tier-1 fast reads first, sorted by (key, term-table
// index), everything else (tier 2, rare shapes, cross list) behind them. A warp's 32 consecutive reads then share their
// key's slot words and neighbouring term-table entries (a few cache lines per gather instead of ~30 — the L1 tag stage
// was what bounded tier 1 once the arithmetic was gone), the state is written in whole lines, tier 1 stops at the last
// fast read, and the delta kernel's reads under one key are neighbours as well. The permutation is applied to the arena's
// read field; the ABI keeps speaking the caller's read ids (gaml_read_values, gaml_cache_save map back).
__global__ void perm_keys_kernel(const uint4* fast, int n, unsigned long long* keys, uint32_t* ids) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const uint4 f = fast[r];
  const bool elsewhere = (f.x >> 31) != 0u, noterm = ((f.x >> 30) & 1u) != 0u;
  unsigned long long k;
  if (elsewhere) k = (1ull << 63) | ((unsigned long long)(f.x & 0x3fffffffu) << 32) | (unsigned long long)f.w;   // tier 2 / cross: by key too
  else if (noterm) k = (0x3fffffffull << 32) | (unsigned long long)(uint32_t)r; // end of the fast region
  else k = ((unsigned long long)(f.x & 0x3fffffffu) << 32) | (unsigned long long)f.w;
  keys[r] = k;
  ids[r] = (uint32_t)r;
}
__global__ void perm_finish_kernel(const unsigned long long* sorted_keys, const uint32_t* sorted_ids, int n, uint32_t* inv, uint32_t* n_fast) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  inv[sorted_ids[i]] = (uint32_t)i;
  const bool here = (sorted_keys[i] >> 63) != 0ull;
  const bool before = i > 0 && (sorted_keys[i - 1] >> 63) != 0ull;
  if (here && !before) *n_fast = (uint32_t)i;   // first read of the "elsewhere" region
  if (i == n - 1 && !here) *n_fast = (uint32_t)n;
}
__global__ void remap_arena_kernel(int4* arena, size_t n, const uint32_t* inv) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    arena[i].x = (int)inv[arena[i].x];
}
size_t perm_temp_bytes(int n) {
  size_t need = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, need, (const unsigned long long*)nullptr, (unsigned long long*)nullptr, (const uint32_t*)nullptr,
                                  (uint32_t*)nullptr, n);
  return need;
}
// keys / ids: 2 x n each (unsorted half, sorted half); inv: n; n_fast: one uint32 on the device.
cudaError_t build_read_permutation(const void* fast, int n, unsigned long long* keys, uint32_t* ids, uint32_t* inv, uint32_t* n_fast,
                                   void* temp, size_t temp_bytes, cudaStream_t st, int* launches) {
  perm_keys_kernel<<<(n + 255) / 256, 256, 0, st>>>(static_cast<const uint4*>(fast), n, keys, ids);
  size_t need = temp_bytes;
  cudaError_t err = cub::DeviceRadixSort::SortPairs(temp, need, (const unsigned long long*)keys, keys + n, (const uint32_t*)ids, ids + n, n, 0, 64, st);
  if (err != cudaSuccess) return err;
  perm_finish_kernel<<<(n + 255) / 256, 256, 0, st>>>(keys + n, ids + n, n, inv, n_fast);
  (*launches) += 3;
  return cudaGetLastError();
}
void launch_remap_arena(void* arena, size_t n_records, const uint32_t* inv, int sm_count, cudaStream_t st) {
  if (n_records) remap_arena_kernel<<<grid_for(n_records, 256, sm_count, 16), 256, 0, st>>>(static_cast<int4*>(arena), n_records, inv);
}

// flags hold their own exclusive scan now: read r is listed iff offs[r + 1] != offs[r]
__global__ void scatter_flagged_kernel(const uint32_t* offs, int n, uint32_t* list) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const uint32_t o = offs[r];
  if (offs[r + 1] != o) list[o] = (uint32_t)r;
}
// Builds FastPair[n] and the cross list (read ids, ascending); flags: n + 1 uint32 of scratch; *n_cross_dev = flags + n
// afterwards (the scan's total).
cudaError_t build_fast_pairs(const void* pairs, int n, int shift, int ins_n, uint32_t uniform_ll, void* fast, uint32_t* flags, uint32_t* list,
                             void* temp, size_t temp_bytes, cudaStream_t st, int* launches) {
  pack_fast_kernel<<<(n + 1 + 255) / 256, 256, 0, st>>>(static_cast<const uint4*>(pairs), n, shift, ins_n, uniform_ll, static_cast<uint4*>(fast), flags);
  size_t need = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, need, flags, flags, n + 1, st);
  if (need > temp_bytes) return cudaErrorMemoryAllocation;
  cudaError_t err = cub::DeviceScan::ExclusiveSum(temp, need, flags, flags, n + 1, st);
  if (err != cudaSuccess) return err;
  scatter_flagged_kernel<<<(n + 255) / 256, 256, 0, st>>>(flags, n, list);
  (*launches) += 3;
  return cudaGetLastError();
}

// Packs the two dense first-record arrays of a paired set into PackedPair; *bad != 0 afterwards when some record does not
// fit (key >= 2^22 or edit distance > 127) and the set keeps streaming the 16-byte records.
__global__ void pack_pairs_kernel(const int4* first1, const int4* first2, int n, const int32_t* partner12, uint4* out, uint32_t* bad) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const int4 a = ldg4(first1 + r), b = ldg4(first2 + r);
  const bool none1 = a.x < 0, none2 = b.x < 0;
  const uint32_t k1 = none1 ? 0u : (uint32_t)a.x, k2 = none2 ? 0u : (uint32_t)b.x;
  const uint32_t ed1 = (uint32_t)a.z & 0xffffu, ed2 = (uint32_t)b.z & 0xffffu;
  if (k1 > kPackKeyMask || k2 > kPackKeyMask || ed1 > kPackEdMask || ed2 > kPackEdMask) *bad = 1u;
  const uint32_t tier2 = ((((uint32_t)a.z | (uint32_t)b.z) >> 17) & 0x1fffu) != 0u ? 1u : 0u;
  uint4 v;
  v.x = (k1 & kPackKeyMask) | ((ed1 & kPackEdMask) << kPackKeyBits) | ((((uint32_t)a.z >> 30) & 1u) << 29) | ((none1 ? 1u : 0u) << 30) | (tier2 << 31);
  // bit 31 of y: both mates lie under the same key (mate 2's key is the partner of mate 1's): one combined slot gather
  const uint32_t same = (partner12 && !none1 && !none2 && partner12[k1] == (int32_t)k2) ? 1u : 0u;
  v.y = (k2 & kPackKeyMask) | ((ed2 & kPackEdMask) << kPackKeyBits) | ((((uint32_t)b.z >> 30) & 1u) << 29) | ((none2 ? 1u : 0u) << 30) | (same << 31);
  v.z = (uint32_t)a.y;
  v.w = (uint32_t)b.y;
  out[r] = v;
}
// Packs the tier-2 list's classes (1,2), (2,1), (2,2) (see tier2_packed_tiles); *bad != 0 when a record does not fit.
__global__ void pack_tier2_kernel(const int4* cdesc, const RowShort* rows1, const RowShort* rows2, int n_entries, int b1, int b2,
                                  uint32_t cb1_0, uint32_t cb1_1, uint32_t cb1_2, uint32_t cb2_0, uint32_t cb2_1, uint32_t cb2_2,
                                  uint32_t tb0, uint32_t tb1, uint32_t tb2, uint4* out, uint32_t* bad) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_entries) return;
  const int cls = (k >= b1 ? 1 : 0) + (k >= b2 ? 1 : 0);
  const int cb = cls == 0 ? 0 : (cls == 1 ? b1 : b2);
  const uint32_t n_c = (uint32_t)((cls == 0 ? b1 : (cls == 1 ? b2 : n_entries)) - cb);
  const uint32_t j = (uint32_t)(k - cb);
  const int n1 = cls == 0 ? 1 : 2, n2 = cls == 1 ? 1 : 2;
  const uint32_t r1 = (cls == 0 ? cb1_0 : (cls == 1 ? cb1_1 : cb1_2)) + (uint32_t)n1 * j;
  const uint32_t r2 = (cls == 0 ? cb2_0 : (cls == 1 ? cb2_1 : cb2_2)) + (uint32_t)n2 * j;
  const uint32_t tb = cls == 0 ? tb0 : (cls == 1 ? tb1 : tb2);
  bool unfit = false;
  auto pack = [&](const RowShort& rw, uint32_t& a, uint32_t& b) {
    const uint32_t ed = (uint32_t)rw.edor & 0xffffu;
    if (rw.key < 0 || (uint32_t)rw.key > kPackKeyMask || ed > kPackEdMask) unfit = true;
    a = ((uint32_t)rw.key & kPackKeyMask) | ((ed & kPackEdMask) << kPackKeyBits) | ((((uint32_t)rw.edor >> 30) & 1u) << 29);
    b = (uint32_t)rw.pos;
  };
  const int4 dsc = cdesc[k];
  uint4 u0, u1, u2;
  u0.x = (uint32_t)dsc.x; u0.y = (uint32_t)dsc.y; u0.z = u0.w = 0u;
  const RowShort x0 = rows1[r1], x1 = rows1[r1 + (n1 > 1 ? 1 : 0)], y0 = rows2[r2], y1 = rows2[r2 + (n2 > 1 ? 1 : 0)];
  if (cls == 0) {
    pack(x0, u0.z, u0.w); pack(y0, u1.x, u1.y); pack(y1, u1.z, u1.w);
  } else if (cls == 1) {
    pack(y0, u0.z, u0.w); pack(x0, u1.x, u1.y); pack(x1, u1.z, u1.w);
  } else {
    pack(x0, u1.x, u1.y); pack(x1, u1.z, u1.w); pack(y0, u2.x, u2.y); pack(y1, u2.z, u2.w);
    out[tb + 2 * n_c + j] = u2;
  }
  out[tb + j] = u0;
  out[tb + n_c + j] = u1;
  if (unfit) *bad = 1u;
}
void launch_pack_tier2(const void* cdesc, const void* rows1, const void* rows2, const int32_t* class_begin, const uint32_t cbase[2][5],
                       const uint32_t tbase[3], void* out, uint32_t* bad, cudaStream_t st) {
  const int n = class_begin[3];
  if (n > 0)
    pack_tier2_kernel<<<(n + 255) / 256, 256, 0, st>>>(static_cast<const int4*>(cdesc), static_cast<const RowShort*>(rows1),
                                                       static_cast<const RowShort*>(rows2), n, class_begin[1], class_begin[2],
                                                       cbase[0][0], cbase[0][1], cbase[0][2], cbase[1][0], cbase[1][1], cbase[1][2],
                                                       tbase[0], tbase[1], tbase[2], static_cast<uint4*>(out), bad);
}

void launch_pack_pairs(const void* first1, const void* first2, int n, const int32_t* partner12, void* out, uint32_t* bad, cudaStream_t st) {
  if (n > 0)
    pack_pairs_kernel<<<(n + 255) / 256, 256, 0, st>>>(static_cast<const int4*>(first1), static_cast<const int4*>(first2), n,
                                                       partner12, static_cast<uint4*>(out), bad);
}

void launch_cdesc_fill(const uint32_t* list, int n_complex, const uint32_t* lens, const uint32_t* cptr1, const uint32_t* cptr2,
                       void* desc, cudaStream_t st) {
  if (n_complex > 0)
    cdesc_fill_kernel<<<(n_complex + 255) / 256, 256, 0, st>>>(list, n_complex, lens, cptr1, cptr2, static_cast<int4*>(desc));
}

size_t coverage_sort_temp_bytes(unsigned n) {
  size_t need = 0;
  cub::DeviceRadixSort::SortKeys(nullptr, need, (const unsigned long long*)nullptr, (unsigned long long*)nullptr, (int)n);
  return need;
}

cudaError_t launch_coverage(const unsigned long long* keys_in, unsigned long long* keys_sorted, unsigned n, void* temp,
                            size_t temp_bytes, const int* cs_begin, const int* cs, double step, double min_from_start, int* bad,
                            int sm_count, cudaStream_t st) {
  size_t need = temp_bytes;
  cudaError_t err = cub::DeviceRadixSort::SortKeys(temp, need, keys_in, keys_sorted, (int)n, 0, 64, st);
  if (err != cudaSuccess) return err;
  coverage_sweep_kernel<<<grid_for(n, 256, sm_count, 8), 256, 0, st>>>(keys_sorted, n, cs_begin, cs, step, min_from_start, bad);
  return cudaGetLastError();
}

void launch_pacbio_alnprob(const AlnProbParams& A, int sm_count, cudaStream_t st) {
  const int grid = grid_for((size_t)A.n, 128, sm_count, 8);
  pacbio_alnprob_kernel<<<grid, 128, 0, st>>>(A);
}

size_t pacbio_coverage_temp_bytes(uint32_t cap) {
  size_t a = 0, b = 0, c = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, a, (const unsigned long long*)nullptr, (unsigned long long*)nullptr, (const int*)nullptr,
                                  (int*)nullptr, (int)cap);
  cub::DeviceRadixSort::SortKeys(nullptr, b, (const unsigned long long*)nullptr, (unsigned long long*)nullptr, (int)(2 * cap));
  cub::DeviceScan::InclusiveScan(nullptr, c, (const unsigned long long*)nullptr, (unsigned long long*)nullptr, PbSegMax(), (int)cap);
  return std::max(a, std::max(b, c));
}

// ikey/iend/pkey hold 2 x their capacity (unsorted half, sorted half); unused slots are padded with all-ones keys, which
// sort behind every real (walk, position). bad is one int.
// phase 0: everything; 1: emit only (a read-id shard's own intervals, left in ikey / iend for gaml_penalty_export);
// 2: sort + sweep only (ikey / iend / pkey / count hold the union of all shards' intervals: gaml_penalty_import)
cudaError_t launch_pacbio_coverage(const PbCovParams& C, unsigned long long* packed, unsigned long long* run_max, void* temp,
                                   size_t temp_bytes, const int* walk_len, double step, int* bad, int sm_count, cudaStream_t st, int phase) {
  const uint32_t cap = C.cap;
  cudaError_t err = cudaSuccess;
  if (phase != 2) {
    err = cudaMemsetAsync(C.ikey, 0xff, (size_t)cap * 2 * 8, st);
    if (err == cudaSuccess) err = cudaMemsetAsync(C.pkey, 0xff, (size_t)cap * 4 * 8, st);
    if (err == cudaSuccess) err = cudaMemsetAsync(C.count, 0, 4, st);
    if (err == cudaSuccess) err = cudaMemsetAsync(bad, 0, 4, st);
    if (err != cudaSuccess) return err;
    pacbio_cov_emit_kernel<<<grid_for(cap, 256, sm_count, 8), 256, 0, st>>>(C);
    if (phase == 1) return cudaGetLastError();
  }
  unsigned long long* ikey_sorted = C.ikey + cap;
  int* iend_sorted = C.iend + cap;
  unsigned long long* pkey_sorted = C.pkey + 2 * (size_t)cap;
  size_t need = temp_bytes;
  err = cub::DeviceRadixSort::SortPairs(temp, need, (const unsigned long long*)C.ikey, ikey_sorted, (const int*)C.iend, iend_sorted,
                                        (int)cap, 0, 64, st);
  if (err != cudaSuccess) return err;
  pacbio_cov_pack_kernel<<<(cap + 255) / 256, 256, 0, st>>>(ikey_sorted, iend_sorted, packed, cap);
  need = temp_bytes;
  err = cub::DeviceScan::InclusiveScan(temp, need, (const unsigned long long*)packed, run_max, PbSegMax(), (int)cap, st);
  if (err != cudaSuccess) return err;
  need = temp_bytes;
  err = cub::DeviceRadixSort::SortKeys(temp, need, (const unsigned long long*)C.pkey, pkey_sorted, (int)(2 * cap), 0, 64, st);
  if (err != cudaSuccess) return err;
  pacbio_cov_sweep_kernel<<<grid_for(2 * (size_t)cap, 256, sm_count, 8), 256, 0, st>>>(pkey_sorted, ikey_sorted, run_max, C.count, cap,
                                                                                       walk_len, step, bad);
  return cudaGetLastError();
}

void launch_exchange_gather(const unsigned long long* lines, int world, int n_sets, int max_sets, uint32_t epoch,
                            unsigned long long* host_lines, unsigned long long* host_flag, unsigned long long timeout_ns, cudaStream_t st) {
  launch_chain(exchange_gather_kernel, 1, kResultStride * 32, st, true, lines, world, n_sets, max_sets, epoch, host_lines, host_flag, timeout_ns);
}
void launch_reduced_publish(const double* reduced, int n_sets, uint32_t epoch, unsigned long long* host_lines, cudaStream_t st) {
  reduced_publish_kernel<<<1, 32, 0, st>>>(reduced, n_sets, epoch, host_lines);
}

size_t csr_temp_bytes(int n_reads) {
  size_t need = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, need, (uint32_t*)nullptr, (uint32_t*)nullptr, n_reads + 1);
  return need;
}

}  // namespace gaml
