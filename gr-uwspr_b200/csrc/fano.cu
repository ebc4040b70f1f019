// The sequential (Fano) decoder on the device: host/wspr_decode.cc:uwspr_b200_fano (which follows
// lib/Fano.cc:110-252 of the reference) as one __device__ function, and the two kernels built on it.
//
// fano_dev keeps the host decoder's control flow step for step -- one loop iteration per decoder
// cycle, the same forward / tighten / back-up / relax decisions, the same counters (metric, cycles,
// maxnp) and, on a time-out, the same partial path in the node stack -- so every output is the host's
// bit for bit.  Narrowed types, each with its bound:
//   * branch metrics: WSPR_METTAB lies in [-137, 5], so a branch metric (two table entries) lies in
//     [-274, 10] and the cumulative metric gamma of a node (at most 81 branches) in [-22 194, 810].
//     Both are kept as int16 in the node stack and as int32 in registers.
//   * encoder state: uint32.  The host keeps 64 bits, but only the low 32 are ever read (the parity
//     masks are 32-bit and the data bytes are the low 8 bits of a node's state); a shift and an
//     increment/xor of bit 0 never move high bits into the low 32.
//   * threshold: int32.  It moves by at most delta per cycle and never rises above the largest
//     ahead = gamma + metric <= 820, so |threshold| + delta <= (maxcycles*nbits + 1)*delta; the entry
//     points reject arguments for which that product does not fit in int32.  The host's tightening loop
//     `while (ahead >= threshold + delta) threshold += delta` is replaced by its closed form
//     threshold += floor((ahead - threshold) / delta) * delta (same value: ahead >= threshold there),
//     evaluated in uint32 because ahead - threshold may exceed INT32_MAX by up to 820 where the result
//     does not.
//
// Node stack: five 32-bit words per node -- encoder state, gamma | branch << 16, the two sorted branch
// metrics, metric[0] | metric[1] << 16 and metric[2] | metric[3] << 16 -- in shared memory, stored
// word-major with the thread index fastest ([word][node][thread]).  With a block width that is a
// multiple of 32, lane l always hits bank l whatever node it is at, so the random per-thread stack
// depths never cause bank conflicts.  82 nodes x 20 bytes x 64 threads + the 1 KB metric table is
// 106 KB per block: two blocks (128 decoders) per SM.
#include <limits.h>

#include "common.cuh"

namespace {

const int kThreads = 64;          // decoders per block (a multiple of 32, see the stack layout above)
const int kNodes = 82;            // nbits + 1 for the largest nbits (81)
const int kWords = 5;             // node stack words per node
// a task of the candidate kernel polls its candidate's first success every kPoll decoder cycles: a
// time-out is 810 000 cycles, so a task made useless by an earlier jiggle's success stops within
// 1/800 of that, at the cost of one L2 load per 1024 cycles
const uint32_t kPoll = 1024;
const uint32_t kPoly1 = 0xf2d05351u;  // Layland-Lushbaugh polynomials, lib/Fano.cc:54-55
const uint32_t kPoly2 = 0xe4613c47u;
const size_t kSmemBytes = sizeof(short) * 512 + sizeof(uint32_t) * kWords * kNodes * kThreads;

enum { W_STATE = 0, W_GB = 1, W_SORT = 2, W_M01 = 3, W_M23 = 4 };

struct FanoResult {
    int status;  // 0 decoded, -1 time-out, 1 abandoned (candidate kernel: an earlier jiggle decoded)
    uint32_t metric, cycles, maxnp;
};

__device__ __forceinline__ uint32_t &node(uint32_t *nd, int word, int k)
{
    return nd[(word * kNodes + k) * kThreads];
}

__device__ __forceinline__ int lo16(uint32_t w) { return (int)(int16_t)(w & 0xffffu); }
__device__ __forceinline__ int hi16(uint32_t w) { return (int)(int16_t)(w >> 16); }
__device__ __forceinline__ uint32_t pack16(int lo, int hi) { return ((uint32_t)lo & 0xffffu) | ((uint32_t)hi << 16); }

// channel symbol pair of an encoder state: POLY1 parity in bit 1, POLY2 parity in bit 0
__device__ __forceinline__ uint32_t branch_pair(uint32_t s)
{
    return ((__popc(s & kPoly1) & 1u) << 1) | (__popc(s & kPoly2) & 1u);
}

// metric[pair] and metric[3 ^ pair] of a node
__device__ __forceinline__ void pair_metrics(uint32_t *nd, int k, uint32_t pair, int &m0, int &m1)
{
    const uint32_t a = node(nd, W_M01, k), b = node(nd, W_M23, k);
    const uint32_t wp = (pair & 2u) ? b : a, wq = (pair & 2u) ? a : b;
    m0 = (pair & 1u) ? hi16(wp) : lo16(wp);
    m1 = (pair & 1u) ? lo16(wq) : hi16(wq);
}

// One decode.  nd: this thread's column of the node stack; sym(p) the p-th de-interleaved soft symbol
// (p < 2*nbits); mt the metric table in shared memory.  With stop != nullptr the decode gives up
// (status 1) once *stop < my_t.
template <typename Sym>
__device__ FanoResult fano_dev(uint32_t *nd, const short *mt, Sym sym, int nbits, int delta, uint32_t maxcycles,
                               const int *stop, int my_t)
{
    const int last = nbits - 1, tail = nbits - 31;
    for (int k = 0; k <= nbits; k++) {
        int m[4] = { 0, 0, 0, 0 };
        if (k <= last) {
            const int a = sym(2 * k), b = sym(2 * k + 1);
            m[0] = mt[a] + mt[b];
            m[1] = mt[a] + mt[256 + b];
            m[2] = mt[256 + a] + mt[b];
            m[3] = mt[256 + a] + mt[256 + b];
        }
        node(nd, W_STATE, k) = 0;
        node(nd, W_GB, k) = 0;
        node(nd, W_SORT, k) = 0;
        node(nd, W_M01, k) = pack16(m[0], m[1]);
        node(nd, W_M23, k) = pack16(m[2], m[3]);
    }
    int np = 0;
    uint32_t deepest = 0;
    {
        int m0, m1;
        pair_metrics(nd, 0, 0u, m0, m1);  // node 0: state 0, pair 0
        if (m0 > m1) {
            node(nd, W_SORT, 0) = pack16(m0, m1);
        } else {
            node(nd, W_SORT, 0) = pack16(m1, m0);
            node(nd, W_STATE, 0) = 1u;
        }
    }
    const uint32_t limit = maxcycles * (uint32_t)nbits;  // < 2^31: checked by the entry points
    int threshold = 0;
    uint32_t i;
    for (i = 1; i <= limit; i++) {
        if (np > (int)deepest) deepest = (uint32_t)np;
        if (stop && (i & (kPoll - 1)) == 0 && *(volatile const int *)stop < my_t) return FanoResult{ 1, 0, 0, 0 };
        const uint32_t gb = node(nd, W_GB, np), so = node(nd, W_SORT, np);
        const int gamma = lo16(gb);
        const int ahead = gamma + ((gb >> 16) ? hi16(so) : lo16(so));
        if (ahead >= threshold) {
            // the node is acceptable; on a first visit tighten the threshold
            if (gamma < threshold + delta && ahead >= threshold + delta)
                threshold = (int)((uint32_t)threshold +
                                  ((uint32_t)ahead - (uint32_t)threshold) / (uint32_t)delta * (uint32_t)delta);
            uint32_t s = node(nd, W_STATE, np) << 1;
            ++np;
            node(nd, W_GB, np) = (uint32_t)ahead & 0xffffu;  // gamma = ahead, branch = 0
            if (np == nbits) {
                node(nd, W_STATE, np) = s;
                break;
            }
            int m0, m1;
            pair_metrics(nd, np, branch_pair(s), m0, m1);
            if (np >= tail) {
                node(nd, W_SORT, np) = (uint32_t)m0 & 0xffffu;  // the tail is all zeros: no 1-branch
            } else if (m0 > m1) {
                node(nd, W_SORT, np) = pack16(m0, m1);
            } else {
                node(nd, W_SORT, np) = pack16(m1, m0);
                s++;  // the 1-branch is the better one
            }
            node(nd, W_STATE, np) = s;
            continue;
        }
        // threshold violated: back up until a node offers an untried second branch
        for (;;) {
            if (np == 0 || lo16(node(nd, W_GB, np - 1)) < threshold) {
                threshold -= delta;  // cannot back up: relax and retry the best branch
                const uint32_t w = node(nd, W_GB, np);
                if (w >> 16) {
                    node(nd, W_GB, np) = w & 0xffffu;
                    node(nd, W_STATE, np) ^= 1u;
                }
                break;
            }
            --np;
            // both words of node np through one address: nvcc 12.9 (ptxas, sm_100a) addressed the state word of
            // node np - 1 here when each word was indexed from np on its own (the PTX was right, the SASS was not)
            uint32_t *const c = &node(nd, W_STATE, np);
            const uint32_t w = c[W_GB * kNodes * kThreads];
            if (np < tail && (w >> 16) != 1u) {
                c[W_GB * kNodes * kThreads] = w | 0x10000u;
                c[0] ^= 1u;
                break;
            }
        }
    }
    FanoResult r;
    r.metric = (uint32_t)lo16(node(nd, W_GB, np));
    r.maxnp = deepest;
    r.cycles = i + 1;
    r.status = (i >= limit) ? -1 : 0;
    return r;
}

__device__ __forceinline__ void load_mettab(short *mt, const short *mettab)
{
    for (int q = threadIdx.x; q < 512; q += blockDim.x) mt[q] = mettab[q];
    __syncthreads();
}

// Task list of the candidate form: one entry g*jig_count + t per (candidate g, jiggle t) with
// worth_a_try && gate, in (g, t) order; also resets first_ok and the task cursor.  One block: an
// exclusive scan of per-thread task counts, as k_worklist does for the candidate list.
__global__ void __launch_bounds__(1024)
k_fano_worklist(const uwspr_b200_refined_t *__restrict__ refined, const uwspr_b200_jiggle_t *__restrict__ jig, int ncand,
                int jig_count, int *__restrict__ first_ok, int *__restrict__ tasks, int *__restrict__ counters)
{
    __shared__ int part[1024];
    const int tid = threadIdx.x;
    const int per = (ncand + 1023) / 1024;
    const int lo = min(ncand, tid * per), hi = min(ncand, lo + per);
    int s = 0;
    for (int g = lo; g < hi; g++) {
        first_ok[g] = INT_MAX;
        if (!refined[g].worth_a_try) continue;
        for (int t = 0; t < jig_count; t++) s += jig[(long long)g * jig_count + t].gate != 0;
    }
    part[tid] = s;
    __syncthreads();
    for (int off = 1; off < 1024; off <<= 1) {
        const int v = (tid >= off) ? part[tid - off] : 0;
        __syncthreads();
        part[tid] += v;
        __syncthreads();
    }
    int run = part[tid] - s;
    for (int g = lo; g < hi; g++) {
        if (!refined[g].worth_a_try) continue;
        for (int t = 0; t < jig_count; t++)
            if (jig[(long long)g * jig_count + t].gate) tasks[run++] = g * jig_count + t;
    }
    if (tid == 1023) {
        counters[0] = part[1023];  // tasks
        counters[1] = 0;           // cursor
    }
}

// Candidate form: each thread takes tasks from a shared cursor until none is left (decode times range
// from ~100 to 810 000 cycles, so a static split would leave most lanes idle behind the time-outs).
//
// Exact early stop.  The host walks t = 0, 1, ... over the gated jiggles of a candidate and stops at
// the first success t*; decoded, idt_used (= t*), the message (t*'s data) and fano_cycles (the sum over
// gated t <= t*) therefore depend only on the tasks with t <= t*.  Here all of a candidate's tasks run
// concurrently; a task that decodes records t in first_ok[g] with atomicMin, so first_ok[g] >= t* at all
// times and it equals t* once t*'s task has finished.  A task gives up only when first_ok[g] < its own
// t, which implies t > t*: no task with t <= t* is ever abandoned, every such task writes its cycles
// (and t*'s task its message), and the reduction reads nothing else.
__global__ void __launch_bounds__(kThreads)
k_fano_tasks(const int *__restrict__ tasks, int *__restrict__ counters, const uint8_t *__restrict__ soft, int jig_count,
             const short *__restrict__ mettab, int *first_ok, uint32_t *__restrict__ task_cycles,
             unsigned long long *__restrict__ task_msg)
{
    extern __shared__ __align__(16) uint32_t smem_fano[];
    short *mt = reinterpret_cast<short *>(smem_fano);
    uint32_t *nd = smem_fano + 256 + threadIdx.x;
    __shared__ uint8_t order[UW_NSYM];   // de-interleaving order: p -> source index (8-bit bit reversal)
    if (threadIdx.x == 0) {
        int p = 0;
        for (int i = 0; p < UW_NSYM && i < 256; i++) {
            const int j = (int)(__brev((uint32_t)i) >> 24);
            if (j < UW_NSYM) order[p++] = (uint8_t)j;
        }
    }
    load_mettab(mt, mettab);
    const int ntasks = counters[0];
    for (;;) {
        const int q = atomicAdd(&counters[1], 1);
        if (q >= ntasks) break;
        const int code = tasks[q];
        const int g = code / jig_count, t = code - g * jig_count;
        if (*(volatile const int *)&first_ok[g] < t) continue;
        const uint8_t *s = soft + (long long)code * UW_NSYM;
        const FanoResult r = fano_dev(nd, mt, [&](int p) { return (int)s[order[p]]; }, 81, 60, 10000u, &first_ok[g], t);
        if (r.status == 1) continue;
        task_cycles[code] = r.cycles;
        if (r.status == 0) {
            unsigned long long m = 0;
            for (int b = 0; b < 7; b++) m |= (unsigned long long)(node(nd, W_STATE, 7 + 8 * b) & 0xffu) << (8 * b);
            task_msg[code] = m;
            atomicMin(&first_ok[g], t);
        }
    }
}

// per-candidate outputs, exactly as uwspr_b200_decode_candidate forms them
__global__ void k_fano_reduce(const uwspr_b200_refined_t *__restrict__ refined, const uwspr_b200_jiggle_t *__restrict__ jig,
                              int ncand, int jig_count, const int *__restrict__ first_ok,
                              const uint32_t *__restrict__ task_cycles, const unsigned long long *__restrict__ task_msg,
                              uint8_t *__restrict__ decoded, int8_t *__restrict__ msg7, int32_t *__restrict__ idt_used,
                              uint32_t *__restrict__ fano_cycles)
{
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= ncand) return;
    int idt = -1;
    uint32_t cyc = 0;
    unsigned long long m = 0;
    if (refined[g].worth_a_try) {
        const int fo = first_ok[g];
        for (int t = 0; t < jig_count && t <= fo; t++)
            if (jig[(long long)g * jig_count + t].gate) cyc += task_cycles[(long long)g * jig_count + t];
        if (fo < jig_count) {
            idt = fo;
            m = task_msg[(long long)g * jig_count + fo];
        }
    }
    decoded[g] = idt >= 0 ? 1 : 0;
    for (int b = 0; b < 7; b++) msg7[(long long)g * 7 + b] = (int8_t)(m >> (8 * b));
    idt_used[g] = idt;
    fano_cycles[g] = cyc;
}

// Raw form: row r of symbols (162 bytes, already de-interleaved) -> the outputs of uwspr_b200_fano.
__global__ void __launch_bounds__(kThreads)
k_fano_rows(const uint8_t *__restrict__ symbols, int n, int nbits, int delta, uint32_t maxcycles,
            const short *__restrict__ mettab, int32_t *__restrict__ status, uint32_t *__restrict__ metric,
            uint32_t *__restrict__ cycles, uint32_t *__restrict__ maxnp, uint8_t *__restrict__ data11)
{
    extern __shared__ __align__(16) uint32_t smem_fano[];
    short *mt = reinterpret_cast<short *>(smem_fano);
    uint32_t *nd = smem_fano + 256 + threadIdx.x;
    load_mettab(mt, mettab);
    const int row = blockIdx.x * kThreads + threadIdx.x;
    if (row >= n) return;
    const uint8_t *s = symbols + (long long)row * UW_NSYM;
    const FanoResult r = fano_dev(nd, mt, [&](int p) { return (int)s[p]; }, nbits, delta, maxcycles, nullptr, 0);
    status[row] = r.status;
    metric[row] = r.metric;
    cycles[row] = r.cycles;
    maxnp[row] = r.maxnp;
    const int nbytes = nbits >> 3;
    for (int b = 0; b < 11; b++)
        data11[(long long)row * 11 + b] = b < nbytes ? (uint8_t)node(nd, W_STATE, 7 + 8 * b) : (uint8_t)0;
}

}  // namespace

int uw_fano_setup()
{
    if (cudaFuncSetAttribute(k_fano_tasks, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes) != cudaSuccess) return 1;
    if (cudaFuncSetAttribute(k_fano_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes) != cudaSuccess) return 1;
    return 0;
}

int uw_fano_blocks_per_sm()
{
    int n = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k_fano_tasks, kThreads, kSmemBytes);
    return n > 0 ? n : 1;
}

void uw_launch_fano_candidates(const uwspr_b200_refined_t *refined, const uwspr_b200_jiggle_t *jig, const uint8_t *soft,
                               int ncand, int jig_count, const short *mettab, int *first_ok, int *tasks, int *counters,
                               uint32_t *task_cycles, unsigned long long *task_msg, int grid, uint8_t *decoded,
                               int8_t *msg7, int32_t *idt_used, uint32_t *fano_cycles, cudaStream_t s)
{
    k_fano_worklist<<<1, 1024, 0, s>>>(refined, jig, ncand, jig_count, first_ok, tasks, counters);
    if (jig_count > 0)
        k_fano_tasks<<<grid, kThreads, kSmemBytes, s>>>(tasks, counters, soft, jig_count, mettab, first_ok, task_cycles, task_msg);
    k_fano_reduce<<<(ncand + 255) / 256, 256, 0, s>>>(refined, jig, ncand, jig_count, first_ok, task_cycles, task_msg, decoded,
                                                      msg7, idt_used, fano_cycles);
}

void uw_launch_fano_rows(const uint8_t *symbols, int n, int nbits, int delta, uint32_t maxcycles, const short *mettab,
                         int32_t *status, uint32_t *metric, uint32_t *cycles, uint32_t *maxnp, uint8_t *data11, cudaStream_t s)
{
    k_fano_rows<<<(n + kThreads - 1) / kThreads, kThreads, kSmemBytes, s>>>(symbols, n, nbits, delta, maxcycles, mettab, status,
                                                                            metric, cycles, maxnp, data11);
}
