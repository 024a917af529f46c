// CUDA backend (sm_100a) of the aeonflux_b200 batch engine: the __global__ wrappers around the stage bodies of
// engine.cuh, their launch geometry, and the C ABI (api_impl.inc).
//
// Geometry: every stage is "one thread per (item, job)" with items along x, so a warp always runs one job type on 32
// consecutive items: control flow is warp-uniform (all data-dependent choices are public digits) and every global
// access is a 128-bit load/store of an item-contiguous record.  Work is integer-multiply bound (IMAD.WIDE on the fma
// pipe); there is no GEMM-shaped step, so no tensor cores, and HBM traffic is ~20 KB per presentation.
#include <cuda_runtime.h>
#include <atomic>

#include <cstdio>
#include <cstdlib>
#include <sched.h>
#include <sys/random.h>

#include "engine.cuh"

namespace afx {

constexpr int TPB = 128;            // threads per CTA for the ladder kernels (4 warps, one per SMSP)
#ifndef AFX_TPB_MSM
#define AFX_TPB_MSM 256
#define AFX_MSM_MINB 2
#endif
// Ladder CTAs run in lockstep (a barrier per ladder step) so that their warps share instruction-cache lines.  Measured on
// B200 (README-4, fused ladders): 1 x 512 threads/SM 24.4 ms, 2 x 256 23.6 ms (finer tail), 4 x 128 25.7 ms (I-cache misses return).
constexpr int TPB_MSM = AFX_TPB_MSM;
constexpr size_t LADDER_SMEM_BUDGET = (size_t)(200 / AFX_MSM_MINB) * 1024;   // per CTA, so that AFX_MSM_MINB CTAs fit one SM

__global__ void __launch_bounds__(256) k_scalar_check(Workspace ws, const u16* fields) {
    u32 item = ws.e_lo + blockIdx.x * blockDim.x + threadIdx.x;
    if (item < ws.e_hi) scalar_check_job(ws, fields[blockIdx.y], item);
}

__global__ void __launch_bounds__(TPB, 4) k_points(Workspace ws, const PointJob* jobs) {
    u32 item = ws.e_lo + blockIdx.x * blockDim.x + threadIdx.x;
    if (item < ws.e_hi) points_job(ws, jobs[blockIdx.y], item);
}

// All ladders of a verify pipeline in ONE launch: the aMAC ladder (when the shape has one) and the constraint MSMs.
// The aMAC ladder is bound by its constant-address table scans (HBM), the MSMs by the IMAD pipe;
// sharing a grid lets the SMs that run aMAC CTAs stream their tables while the others multiply, instead of every SM
// contending for HBM at once.  The one MSM that consumes Z (constraint "Z", presentation.rs:416) is ordered last and waits
// on a per-CTA completion flag written by the aMAC CTAs (release/acquire at gpu scope).
// Work is claimed through an atomic TICKET, not blockIdx: a CTA's position in the block order below is the value it draws from
// a per-launch counter when it starts running.  Every position below a consumer's was therefore drawn by a CTA that is already
// resident and running, so a spinning consumer can only ever wait for producers that are making progress -- whatever order
// the hardware, MPS or a debugger dispatches CTAs in.
__device__ __forceinline__ u32 ld_acquire(const u32* p) { u32 v; asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v; }
__device__ __forceinline__ void st_release(u32* p, u32 v) { asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }

struct LadderArgs {
    const MsmDesc* msms; const u32* group_idx; u32 scratch_terms;
    const AmacDesc* amac;     // nullable
    u32* flags; u32 epoch; u32 flag_tpb; int dep_msm;   // MSM index that must wait for the aMAC CTAs covering its items (-1 none)
    u32* ticket;                    // zeroed on the stream before the launch
    u32 nx, n_ind, n_dep, stride;   // block order, see ladder_block()
};
// Block order of the fused launch (1-D grid).  nx = CTAs per job.  First the n_ind independent MSM jobs (job-major) with one
// aMAC CTA slotted in every `stride` positions, so that at any time only a fraction of the SMs stream aMAC tables; then
// the n_dep jobs that wait on the aMAC flags.  Returns the job (-1 = aMAC, else position in group_idx) and sets bx.
__device__ __forceinline__ int ladder_block(const LadderArgs& a, u32 b, u32& bx) {
    const u32 n_amac = a.amac ? a.nx : 0, head = a.n_ind * a.nx + n_amac;
    if (b >= head) { u32 m = b - head; bx = m % a.nx; return (int)(a.n_ind + m / a.nx); }
    u32 m;
    if (n_amac && b < n_amac * a.stride) {
        if (b % a.stride == 0) { bx = b / a.stride; return -1; }
        m = b - (b / a.stride + 1);
    } else m = b - n_amac;
    bx = m % a.nx;
    return (int)(m / a.nx);
}

__global__ void __launch_bounds__(TPB_MSM, AFX_MSM_MINB) k_ladders(Workspace ws, LadderArgs a) {
    extern __shared__ __align__(16) u32 smem[];
    __shared__ u32 s_ticket;
    if (threadIdx.x == 0) s_ticket = atomicAdd(a.ticket, 1u);
    __syncthreads();
    u32 bx;
    const int job = ladder_block(a, s_ticket, bx);
    u32 item = bx * blockDim.x + threadIdx.x;
    bool active = item < ws.count;
    if (!active) item = ws.count - 1;                              // keep every thread in the barriers of the ladder
    if (job < 0) {
        amac_job(ws, *a.amac, item, smem + threadIdx.x, blockDim.x, active);
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) st_release(a.flags + bx, a.epoch);
        return;
    }
    const u32 y = (u32)job;
    const u32 mi = a.group_idx[y];
    const MsmDesc& d = a.msms[mi];
    u32* scratch = smem;                                            // [scratch_terms*8][TPB_MSM]
    if ((int)mi == a.dep_msm && threadIdx.x == 0) {
        u32 lo = (bx * blockDim.x) / a.flag_tpb;
        u32 last_item = bx * blockDim.x + blockDim.x - 1;
        if (last_item >= ws.count) last_item = ws.count - 1;
        for (u32 f = lo; f <= last_item / a.flag_tpb; f++)
            while (ld_acquire(a.flags + f) != a.epoch) __nanosleep(256);
    }
    __syncthreads();
    CtabResolver ctab_of{ws.ctabs, &d};
    msm_job(ws, d, item, scratch + threadIdx.x, blockDim.x, ctab_of, active);
}

// Small batches: the aMAC ladder cut into parts (engine.cuh:amac_part_job) beside the constraint MSMs that do not need Z -- no job of
// this grid depends on another, so there are no flags and no ticket; k_amac_combine and the "Z" constraint follow in stream order.
struct PartsArgs {
    const MsmDesc* msms; const u32* group_idx; u32 scratch_terms;
    const AmacDesc* amac; u32* parts_out; u32 n_parts, nx;
    AmacPart parts[MAX_AMAC_PARTS];
};
__global__ void __launch_bounds__(TPB_MSM, AFX_MSM_MINB) k_ladders_parts(Workspace ws, PartsArgs a) {
    extern __shared__ __align__(16) u32 smem[];
    const u32 job = blockIdx.x / a.nx, bx = blockIdx.x % a.nx;
    u32 item = bx * blockDim.x + threadIdx.x;
    bool active = item < ws.count;
    if (!active) item = ws.count - 1;
    if (job < a.n_parts) {
        amac_part_job(ws, *a.amac, a.parts[job], a.parts_out + (size_t)job * ws.count * 32, item, smem + threadIdx.x, blockDim.x, active);
        return;
    }
    const MsmDesc& d = a.msms[a.group_idx[job - a.n_parts]];
    CtabResolver ctab_of{ws.ctabs, &d};
    msm_job(ws, d, item, smem + threadIdx.x, blockDim.x, ctab_of, active);
}
__global__ void __launch_bounds__(128) k_amac_combine(Workspace ws, const AmacDesc* d, const u32* parts, u32 n_parts) {
    u32 item = blockIdx.x * blockDim.x + threadIdx.x;
    if (item < ws.count) amac_combine_job(ws, *d, parts, n_parts, item);
}

// Commitment encodings of the verify MSMs (engine.cuh:commit_encode_job): thread (item, y) encodes entries [y * per, y * per + per)
// of the slot list under one inversion
__global__ void __launch_bounds__(128) k_commit_encode(Workspace ws, const u32* slots, u32 nslots, u32 per) {
    u32 item = blockIdx.x * blockDim.x + threadIdx.x;
    const u32 lo = blockIdx.y * per;
    if (item < ws.count) commit_encode_job(ws, slots + lo, nslots - lo < per ? nslots - lo : per, item);
}

// Issuer::issue: the same per-(item, job) ladders with every lookup constant-address (all scalars are secrets)
__global__ void __launch_bounds__(TPB_MSM, AFX_MSM_MINB) k_msm_ct(Workspace ws, const MsmDesc* msms, const u32* group_idx) {
    extern __shared__ __align__(16) u32 smem[];
    const MsmDesc& d = msms[group_idx[blockIdx.y]];
    u32 item = blockIdx.x * blockDim.x + threadIdx.x;
    bool active = item < ws.count;
    if (!active) item = ws.count - 1;
    msm_ct_job(ws, d, item, smem + threadIdx.x, blockDim.x, active);
}

__global__ void __launch_bounds__(256) k_derive(Workspace ws, const DeriveOp* ops, u32 nops) {
    u32 item = blockIdx.x * blockDim.x + threadIdx.x;
    if (item < ws.count) derive_program_job(ws, ops, nops, item);
}

__global__ void __launch_bounds__(256) k_out_words(Workspace ws, const OutWord* d, u32* out) {
    u32 item = blockIdx.x * blockDim.x + threadIdx.x;
    if (item < ws.count) out_word_job(ws, d[blockIdx.y], blockIdx.y, item, out);
}

__global__ void __launch_bounds__(TPB) k_transcript(Workspace ws, const TxDesc* txs) {
    u32 item = blockIdx.x * blockDim.x + threadIdx.x;
    if (item < ws.count) transcript_job(ws, txs[blockIdx.y], item);
}

// ladder table of Z from its extended coordinates (exact fallback of an RLC chunk whose front half skipped the tables)
__global__ void __launch_bounds__(128) k_ztable(Workspace ws, const AmacDesc* d) {
    u32 item = blockIdx.x * blockDim.x + threadIdx.x;
    if (item < ws.count) ztable_job(ws, *d, item);
}

__global__ void __launch_bounds__(256) k_commit_compare(Workspace ws, const CmpPair* pairs) {
    u32 item = blockIdx.x * blockDim.x + threadIdx.x;
    if (item < ws.count) commit_compare_job(ws, pairs[blockIdx.y], item);
}

// ---- random-linear-combination path (BatchableProof): coefficients, Pippenger bucket method, final check -------------------
__global__ void __launch_bounds__(128) k_rlc_scalars(Workspace ws, const RlcDesc* d, RlcBuffers rb) {
    u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < rb.cnt) rlc_scalars_job(ws, *d, rb, rb.lo + i);
}
// one CTA per constant term: chunk-wide sum of its coefficients mod l (9-word partial sums, shared-memory tree)
__global__ void __launch_bounds__(256) k_rlc_colsum(Workspace ws, RlcBuffers rb) {
    __shared__ u32 part[256][9];
    const u32 t = blockIdx.x;
    u32 acc[9];
    for (int i = 0; i < 9; i++) acc[i] = 0;
    for (u32 item = threadIdx.x; item < rb.cnt; item += blockDim.x) {
        u32 v[8]; load8(v, rb.cterm + ((size_t)t * rb.cnt + item) * 8);
        rlc_add288(acc, v);
    }
    for (int i = 0; i < 9; i++) part[threadIdx.x][i] = acc[i];
    __syncthreads();
    for (u32 s = blockDim.x / 2; s > 0; s >>= 1) {
        if (threadIdx.x < s) rlc_add288x(part[threadIdx.x], part[threadIdx.x + s]);
        __syncthreads();
    }
    if (threadIdx.x == 0) { sc r = rlc_reduce288(part[0]); for (int i = 0; i < 8; i++) rb.csum[8 * t + i] = r.v[i]; }
}
__global__ void __launch_bounds__(256) k_rlc_digits(const RlcDesc* d, RlcBuffers rb) {
    u32 n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n < rb.N) rlc_digits_job(*d, rb, n);
}
// one CTA per window: exclusive scan of the 2^(c-1) bucket sizes (each thread owns a run of consecutive buckets; the run
// totals are scanned in shared memory), offsets written in place and copied to the scatter cursors
__global__ void __launch_bounds__(1024) k_rlc_scan(RlcBuffers rb) {
    __shared__ u32 part[1024];
    const u32 w = blockIdx.x, T = blockDim.x, L = (rb.nb + T - 1) / T;
    u32* h = rb.hist + (size_t)w * (rb.nb + 1);
    u32* cur = rb.cursor + (size_t)w * (rb.nb + 1);
    const u32 lo = threadIdx.x * L + 1;
    u32 sum = 0;
    for (u32 b = lo; b < lo + L && b <= rb.nb; b++) sum += h[b];
    part[threadIdx.x] = sum;
    __syncthreads();
    for (u32 d = 1; d < T; d <<= 1) {                      // Hillis-Steele inclusive scan of the run totals
        u32 v = threadIdx.x >= d ? part[threadIdx.x - d] : 0;
        __syncthreads();
        part[threadIdx.x] += v;
        __syncthreads();
    }
    u32 run = part[threadIdx.x] - sum;
    for (u32 b = lo; b < lo + L && b <= rb.nb; b++) { u32 cnt = h[b]; h[b] = run; cur[b] = run; run += cnt; }
    if (threadIdx.x == T - 1) h[0] = part[T - 1];          // total number of non-zero digits of the window
}
__global__ void __launch_bounds__(256) k_rlc_scatter(RlcBuffers rb) {
    u32 n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n < rb.N) rlc_scatter_job(rb, n);
}
__global__ void __launch_bounds__(128, 4) k_rlc_buckets(Workspace ws, const RlcDesc* d, RlcBuffers rb) {
    u32 t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < rb.nwin * rb.nb) rlc_bucket_job(ws, *d, rb, t / rb.nb, t % rb.nb + 1);
}
// sum_b b * B_b of one window per CTA: each thread reduces a segment of buckets by running sums, then the partial sums are
// combined with warp shuffles (a point is 32 words: 32 shuffles per level) and one shared-memory hop between the warps.
__device__ __forceinline__ ge ge_shfl_down(const ge& p, u32 delta) {
    ge r;
    for (int i = 0; i < 8; i++) {
        r.X.v[i] = __shfl_down_sync(0xffffffffu, p.X.v[i], delta); r.Y.v[i] = __shfl_down_sync(0xffffffffu, p.Y.v[i], delta);
        r.Z.v[i] = __shfl_down_sync(0xffffffffu, p.Z.v[i], delta); r.T.v[i] = __shfl_down_sync(0xffffffffu, p.T.v[i], delta);
    }
    return r;
}
__global__ void __launch_bounds__(512) k_rlc_window_reduce(RlcBuffers rb) {
    __shared__ u32 warp_sum[16][32];
    const u32 w = blockIdx.x, T = blockDim.x;
    const u32 L = (rb.nb + T - 1) / T;
    u32 lo = threadIdx.x * L + 1, hi = lo + L - 1;
    if (hi > rb.nb) hi = rb.nb;
    ge acc = lo <= rb.nb ? rlc_segment_job(rb, w, lo, hi) : ge_identity();
    for (u32 delta = 16; delta > 0; delta >>= 1) {
        ge other = ge_shfl_down(acc, delta);
        acc = ge_add(acc, other);              // lanes beyond the live half add garbage that is never read
    }
    if ((threadIdx.x & 31u) == 0) store_ge(warp_sum[threadIdx.x >> 5], acc);
    __syncthreads();
    if (threadIdx.x == 0) {
        ge tot = load_ge(warp_sum[0]);
        for (u32 k = 1; k < T / 32; k++) tot = ge_add(tot, load_ge(warp_sum[k]));
        store_ge(rb.wsum + (size_t)w * 32, tot);
    }
}
// one warp: the lanes share out the generators' fixed-base multiplications (comb tables) while lane 0 also runs the Horner
// pass over the window sums; a shuffle reduction joins them and lane 0 publishes the verdict of the chunk
__global__ void __launch_bounds__(32) k_rlc_final(Workspace ws, const RlcDesc* d, RlcBuffers rb) {
    ge acc = ge_identity();
    for (u32 t = threadIdx.x; t < d->ncterms; t += 32) acc = ge_add(acc, rlc_cterm_point(ws, *d, rb, t));
    if (threadIdx.x == 0) acc = ge_add(acc, rlc_horner(rb));
    for (u32 delta = 16; delta > 0; delta >>= 1) {
        ge other = ge_shfl_down(acc, delta);
        acc = ge_add(acc, other);
    }
    if (threadIdx.x == 0) rlc_publish(rb, acc);
}

__global__ void __launch_bounds__(256) k_verdict(Workspace ws, uint8_t* verdicts) {
    u32 item = blockIdx.x * blockDim.x + threadIdx.x;
    if (item < ws.count) verdicts[item] = ws.status[item] != 0;
}

// Mixed-shape calls: one CTA per tile of BUCKET_TILE records.  Every thread locates one record (engine.cuh:bucket_locate, over the
// tile's ids in shared memory); then each warp copies whole records, its lanes on consecutive 16-byte quads of one record.
__global__ void __launch_bounds__(BUCKET_TILE) k_bucket_records(BucketArgs a) {
    __shared__ uint8_t ids[BUCKET_TILE];
    __shared__ u32 rec_words[256];
    __shared__ u64 src[BUCKET_TILE], dst[BUCKET_TILE];
    const u32 i0 = blockIdx.x * BUCKET_TILE, n = a.count - i0 < BUCKET_TILE ? a.count - i0 : BUCKET_TILE, t = threadIdx.x;
    if (t < n) ids[t] = a.ids[i0 + t];
    if (t < a.n_shapes) rec_words[t] = a.rec_words[t];
    __syncthreads();
    if (t < n) a.slot[i0 + t] = bucket_locate(a, ids, rec_words, i0 + t, src[t], dst[t]);
    __syncthreads();
    for (u32 r = t / 32; r < n; r += BUCKET_TILE / 32) bucket_copy(a.records + src[r], a.fields + dst[r], rec_words[ids[r]], t % 32, 32);
}
// Mixed-shape prover calls, the inverse of k_bucket_records: every thread locates one record's output (engine.cuh:unbucket_locate)
// and scatters its status byte; then each warp copies whole output records back into record order.
__global__ void __launch_bounds__(BUCKET_TILE) k_unbucket_records(UnbucketArgs a) {
    __shared__ uint8_t ids[BUCKET_TILE];
    __shared__ u32 out_words[256];
    __shared__ u64 src[BUCKET_TILE], dst[BUCKET_TILE];
    const u32 i0 = blockIdx.x * BUCKET_TILE, n = a.count - i0 < BUCKET_TILE ? a.count - i0 : BUCKET_TILE, t = threadIdx.x;
    if (t < n) ids[t] = a.ids[i0 + t];
    if (t < a.n_shapes) out_words[t] = a.out_words[t];
    __syncthreads();
    if (t < n) a.status[i0 + t] = unbucket_locate(a, ids, out_words, i0 + t, src[t], dst[t]);
    __syncthreads();
    for (u32 r = t / 32; r < n; r += BUCKET_TILE / 32) bucket_copy(a.outputs + src[r], a.records + dst[r], out_words[ids[r]], t % 32, 32);
}

// per-issuer setup: one thread per (constant point, multiple)
__global__ void __launch_bounds__(128) k_ctab_setup(const u32* enc, u32 ncp, u32* ctabs, u32* encneg, u32* bad, u32 entries, int bits) {
    u32 t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= ncp * entries) return;
    u32 b = t / entries, m = t % entries + 1;
    u32 ok = ctab_entry_job(enc + 8 * b, m, ctabs + ((size_t)b * entries + (m - 1)) * 24, bits + 1);
    if (m == 1) {
        ge p; u32 w[8];
        ge_decompress(p, enc + 8 * b);
        ge_compress(w, ge_neg(p));
        for (int i = 0; i < 8; i++) encneg[8 * b + i] = w[i];
        if (!ok) atomicOr(bad, 1u);
    }
}
__global__ void __launch_bounds__(128) k_comb_setup(const u32* enc, u32 ncp, u32* comb) {
    u32 t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= ncp * COMB_WINDOWS * COMB_ENTRIES) return;
    u32 b = t / (COMB_WINDOWS * COMB_ENTRIES), r = t % (COMB_WINDOWS * COMB_ENTRIES);
    comb_entry_job(enc + 8 * b, r / COMB_ENTRIES, r % COMB_ENTRIES + 1, comb + (size_t)t * 24);
}
__global__ void __launch_bounds__(32) k_link_setup(const u32* enc_gy, u32 ny, u32* out) {
    u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 1 && i < ny) link_entry_job(enc_gy, i, out + 8 * i);
}
__global__ void __launch_bounds__(128) k_primitive(u32 op, const u32* in, u32* out, u32* flags, u32 count) {
    u32 item = blockIdx.x * blockDim.x + threadIdx.x;
    if (item < count) primitive_job(op, in, out, flags, item);
}
// symmetric encryption of attributes: one thread per item (engine.cuh:encode_job / decrypt_job)
__global__ void __launch_bounds__(128) k_encode(const uint8_t* data, u32* pt, uint8_t* status, u32 count, u32 item_major) {
    u32 item = blockIdx.x * blockDim.x + threadIdx.x;
    if (item < count) encode_job(data, pt, status, count, item_major, item);
}
__global__ void __launch_bounds__(128) k_decrypt(const u32* ct, const u32* kp, u32* tabs, uint8_t* data, u32* pt, uint8_t* status, u32 count,
                                                 u32 item_major) {
    u32 item = blockIdx.x * blockDim.x + threadIdx.x;
    if (item < count) decrypt_job(ct, kp, tabs, data, pt, status, count, item_major, item);
}
// Keypair::derive: the three hashes and wide reductions, one thread per item (engine.cuh:keypair_scalars_job); pk is compile_keypair
__global__ void __launch_bounds__(128) k_keypair_scalars(const u32* ms, u32* rows, u32 count) {
    u32 item = blockIdx.x * blockDim.x + threadIdx.x;
    if (item < count) keypair_scalars_job(ms, rows, count, item);
}
__global__ void k_secret_setup(const u32* secsc, u32 nsec, u32* secdig, const u32* Wenc, u32* W_pniels, u32* bad) {
    u32 t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < nsec) {
        sc s = sc_from_words(secsc + 8 * t);
        if (!sc_is_canonical(s)) atomicOr(bad, 2u);
        u32 rec[8]; sc_recode16(rec, s);
        for (int i = 0; i < 8; i++) secdig[8 * t + i] = rec[i];
    } else if (t == nsec) {
        ge p;
        if (!ge_decompress(p, Wenc)) atomicOr(bad, 1u);
        store_pniels(W_pniels, ge_to_pniels(p));
    }
}

}  // namespace afx

// ---- backend primitives for api_impl.inc -------------------------------------------------------------------------------
using namespace afx;
typedef cudaStream_t be_stream;
#define AFX_BACKEND_NAME "cuda sm_100a"

static int be_set_device(int d) { return cudaSetDevice(d) != cudaSuccess; }
static int be_malloc(void** p, size_t n) { return cudaMalloc(p, n ? n : 16) != cudaSuccess; }
static void be_free(void* p) { cudaFree(p); }
static int be_h2d(void* d, const void* h, size_t n, be_stream s) { return cudaMemcpyAsync(d, h, n, cudaMemcpyHostToDevice, s) != cudaSuccess; }
static int be_d2h(void* h, const void* d, size_t n, be_stream s) { return cudaMemcpyAsync(h, d, n, cudaMemcpyDeviceToHost, s) != cudaSuccess; }
static int be_d2d(void* d, const void* src, size_t n, be_stream s) { return cudaMemcpyAsync(d, src, n, cudaMemcpyDeviceToDevice, s) != cudaSuccess; }
static int be_memset(void* d, int v, size_t n, be_stream s) { return cudaMemsetAsync(d, v, n, s) != cudaSuccess; }
static int be_sync(be_stream s) { return cudaStreamSynchronize(s) != cudaSuccess; }
static int be_check_launch() {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { std::fprintf(stderr, "aeonflux_b200: CUDA launch failed: %s\n", cudaGetErrorString(e)); return -3; }
    return 0;
}
static int be_os_random(void* p, size_t n) { return getrandom(p, n, 0) != (ssize_t)n; }
// Pin the calling thread to the CPUs of the NUMA node the device hangs off (sysfs local_cpulist of its PCI function), so that the
// page-locked staging it allocates next is node-local and its copies do not cross the socket interconnect.  Best effort: returns
// non-zero and changes nothing when the topology cannot be read.
static int be_bind_thread_to_device(int device) {
    char bus[32] = {0};
    if (cudaDeviceGetPCIBusId(bus, sizeof bus, device) != cudaSuccess) return 1;
    for (char* p = bus; *p; p++) if (*p >= 'A' && *p <= 'F') *p = (char)(*p - 'A' + 'a');
    char path[128];
    std::snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/local_cpulist", bus);
    FILE* f = std::fopen(path, "r");
    if (!f) return 1;
    char list[4096] = {0};
    size_t got = std::fread(list, 1, sizeof list - 1, f);
    std::fclose(f);
    if (!got) return 1;
    cpu_set_t set; CPU_ZERO(&set);
    int any = 0;
    for (char* p = list; *p;) {
        char* end;
        long a = std::strtol(p, &end, 10), b = a;
        if (end == p) break;
        if (*end == '-') { p = end + 1; b = std::strtol(p, &end, 10); }
        for (long c = a; c <= b && c < CPU_SETSIZE; c++) { CPU_SET((int)c, &set); any = 1; }
        p = (*end == ',') ? end + 1 : end;
        if (*end != ',' ) break;
    }
    if (!any) return 1;
    return sched_setaffinity(0, sizeof set, &set) != 0;
}
static size_t be_split_copy_min_items() { return 8192; }     // below this a call is launch-bound and one copy is as good
typedef cudaEvent_t be_event;
static void be_event_create(be_event* e) { cudaEventCreate(e); }
static void be_event_destroy(be_event e) { cudaEventDestroy(e); }
static void be_event_record(be_event e, be_stream s) { cudaEventRecord(e, s); }
static int be_event_sync(be_event e) { return cudaEventSynchronize(e) != cudaSuccess; }
static float be_event_elapsed(be_event a, be_event b) { float ms = 0; cudaEventElapsedTime(&ms, a, b); return ms; }
static int be_stream_create(be_stream* s) { return cudaStreamCreateWithFlags(s, cudaStreamNonBlocking) != cudaSuccess; }
static void be_stream_destroy(be_stream s) { cudaStreamDestroy(s); }
static void be_stream_wait(be_stream s, be_event e) { cudaStreamWaitEvent(s, e, 0); }
static int be_host_alloc(void** p, size_t n) { return cudaHostAlloc(p, n, cudaHostAllocDefault) != cudaSuccess; }
static void be_host_free(void* p) { cudaFreeHost(p); }
static dim3 grid_for(u32 count, u32 tpb, u32 y) { return dim3((count + tpb - 1) / tpb, y, 1); }

static void be_launch_scalar_check(const Workspace& ws, const u16* d_fields, u32 nf, be_stream s) {
    k_scalar_check<<<grid_for(ws.e_hi - ws.e_lo, 256, nf), 256, 0, s>>>(ws, d_fields);
}
static void be_launch_points(const Workspace& ws, const PointJob* d_jobs, u32 njobs, be_stream s) {
    k_points<<<grid_for(ws.e_hi - ws.e_lo, TPB, njobs), TPB, 0, s>>>(ws, d_jobs);
}
// The opt-in to > 48 KiB of dynamic shared memory is a per-device function attribute: set it once per (kernel, device).
static int sm_count() {
    static std::atomic<int> cached[64];
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) return 148;
    int n = cached[dev].load(std::memory_order_relaxed);
    if (n == 0) {
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached[dev].store(n, std::memory_order_relaxed);
    }
    return n;
}
static void allow_large_smem(const void* kernel, int which) {
    static std::atomic<bool> done[3][64];          // contexts on different devices are driven from different host threads
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || !done[which][dev].load(std::memory_order_acquire)) {
        cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024);
        if (dev >= 0 && dev < 64) done[which][dev].store(true, std::memory_order_release);
    }
}

// Launch geometry of a ladder kernel whose CTAs hold `terms` terms of digit scratch: the largest CTA (<= TPB_MSM threads) whose
// scratch fits LADDER_SMEM_BUDGET, and that scratch in bytes.
struct LadderGeometry { u32 tpb; size_t smem; };
static LadderGeometry ladder_geometry(u32 terms) {
    u32 tpb = TPB_MSM;
    size_t smem = 0;
    for (;; tpb /= 2) {
        smem = (size_t)terms * 8 * tpb * 4;
        if (smem <= LADDER_SMEM_BUDGET || tpb <= 32) break;
    }
    return {tpb, smem};
}

// One launch for the aMAC ladder (if `amac`) plus the MSMs of one scratch-size group.
// The last n_dep_jobs entries of d_idx are the MSMs that wait on the aMAC flags.
static u32 be_launch_ladders(const Workspace& ws, const AmacDesc* amac, u32 amac_nps, const MsmDesc* d_msms, const u32* d_idx, u32 nidx, u32 n_dep_jobs,
                             u32 max_terms, u32 amac_terms, int dep_msm, u32* flags, u32 epoch, u32 flag_tpb, u32* ticket, be_stream s) {
    u32 terms = max_terms > amac_nps ? max_terms : amac_nps;
    const auto [tpb, smem] = ladder_geometry(terms);
    allow_large_smem((const void*)k_ladders, 0);
    const u32 nx = (ws.count + tpb - 1) / tpb;
    const u32 n_dep = n_dep_jobs < nidx ? n_dep_jobs : nidx, n_ind = nidx - n_dep;
    const u32 head = n_ind * nx + (amac ? nx : 0);
    // aMAC CTAs are spread over the first part of the independent work (one per `stride` positions) so that only a fraction of the SMs
    // stream aMAC tables at any time: the first 70 % when the launch is many waves long (README-4, 65,536 items: 50 % 21.32 ms, 70 %
    // 21.34, 90 % 22.46, 100 % 23.87).  But an aMAC CTA runs `a_rel` times as long as a constraint CTA (2 + n bases, scans) and the "Z"
    // constraint waits for it, so the last one has to START a_rel + 1.5 CTA-durations before the grid would otherwise end -- in a
    // short launch that means earlier than 70 %, down to "all aMAC CTAs first".  ms per synchronous call, fixed 70 % -> this rule:
    // README-4 16,384 items 9.97 -> 8.16, 32,768: 14.11 -> 13.07, 65,536: 25.17 -> 25.15; S16 16,384: 33.3 -> 29.5, 32,768: 66.8 -> 59.2,
    // 65,536: 117.2 -> 116.9 (the estimate's two constants were varied by +-40 %: no difference).
    u32 stride = 1;
    if (amac) {
        const double a_rel = (99.0 + 37.0 * amac_terms) / 140.0;
        const double waves = ((double)n_ind * nx + a_rel * nx + (double)n_dep * nx) / (2.0 * sm_count());
        double frac = (waves - a_rel - 1.5) / waves;
        if (frac > 0.7) frac = 0.7;
        if (frac > 0) stride = (u32)((double)head * frac / nx);
        // ... but never shoulder to shoulder: consecutive positions land on neighbouring SMs, and a GPC full of table-scanning CTAs is
        // slower than the same CTAs spread over the chip (4,096 S16 items, unsplit: 15.3 ms spread, 16.8 ms packed).  Inside the
        // first wave a stride costs no start time.
        u32 spread = (u32)(2 * sm_count()) / nx, cap = (u32)((uint64_t)head * 7 / 10 / nx);
        if (spread > cap) spread = cap;
        if (stride < spread) stride = spread;
        if (stride < 1) stride = 1;
    }
    LadderArgs a{d_msms, d_idx, terms, amac, flags, epoch, amac ? tpb : flag_tpb, dep_msm, ticket, nx, n_ind, n_dep, stride};
    cudaMemsetAsync(ticket, 0, 4, s);
    k_ladders<<<nx * (nidx + (amac ? 1 : 0)), tpb, smem, s>>>(ws, a);
    return tpb;
}
static void be_launch_ladders_parts(const Workspace& ws, const AmacDesc* amac, const AmacPart* parts, u32 n_parts, u32 part_terms, u32* parts_out,
                                    const MsmDesc* d_msms, const u32* d_idx, u32 nidx, u32 max_terms, be_stream s) {
    u32 terms = max_terms > part_terms ? max_terms : part_terms;
    if (terms < 1) terms = 1;
    const auto [tpb, smem] = ladder_geometry(terms);
    allow_large_smem((const void*)k_ladders_parts, 2);
    PartsArgs a;
    a.msms = d_msms; a.group_idx = d_idx; a.scratch_terms = terms; a.amac = amac; a.parts_out = parts_out; a.n_parts = n_parts;
    a.nx = (ws.count + tpb - 1) / tpb;
    for (u32 k = 0; k < (u32)MAX_AMAC_PARTS; k++) a.parts[k] = k < n_parts ? parts[k] : AmacPart{0, 0, 0, 0};
    k_ladders_parts<<<a.nx * (n_parts + nidx), tpb, smem, s>>>(ws, a);
}
static void be_launch_amac_combine(const Workspace& ws, const AmacDesc* amac, const u32* parts_out, u32 n_parts, be_stream s) {
    k_amac_combine<<<grid_for(ws.count, 128, 1), 128, 0, s>>>(ws, amac, parts_out, n_parts);
}
static void be_launch_commit_encode(const Workspace& ws, const u32* d_slots, u32 nslots, u32 per, be_stream s) {
    k_commit_encode<<<grid_for(ws.count, 128, (nslots + per - 1) / per), 128, 0, s>>>(ws, d_slots, nslots, per);
}
static void be_launch_msm_ct(const Workspace& ws, const MsmDesc* d_msms, const u32* d_idx, u32 nidx, u32 max_terms, be_stream s) {
    const auto [tpb, smem] = ladder_geometry(max_terms);
    allow_large_smem((const void*)k_msm_ct, 1);
    k_msm_ct<<<grid_for(ws.count, tpb, nidx), tpb, smem, s>>>(ws, d_msms, d_idx);
}
static void be_launch_derive(const Workspace& ws, const DeriveOp* d, u32 nd, be_stream s) {
    k_derive<<<grid_for(ws.count, 256, 1), 256, 0, s>>>(ws, d, nd);
}
static void be_launch_out_words(const Workspace& ws, const OutWord* d, u32 nwords, u32* out, be_stream s) {
    k_out_words<<<grid_for(ws.count, 256, nwords), 256, 0, s>>>(ws, d, out);
}
static void be_launch_transcript(const Workspace& ws, const TxDesc* d_txs, u32 ntx, be_stream s) {
    k_transcript<<<grid_for(ws.count, TPB, ntx), TPB, 0, s>>>(ws, d_txs);
}
static void be_launch_ztable(const Workspace& ws, const AmacDesc* d, be_stream s) { k_ztable<<<grid_for(ws.count, 128, 1), 128, 0, s>>>(ws, d); }
static void be_launch_commit_compare(const Workspace& ws, const CmpPair* d_pairs, u32 npairs, be_stream s) {
    k_commit_compare<<<grid_for(ws.count, 256, npairs), 256, 0, s>>>(ws, d_pairs);
}
// The whole RLC pass of one chunk: coefficients, column sums, Pippenger, final check.  8 launches.
static u32 be_launch_rlc(const Workspace& ws, const RlcDesc* d_desc, u32 ncterms, const RlcBuffers& rb, be_stream s, be_event* ev_bucket = nullptr) {
    cudaMemsetAsync(rb.hist, 0, (size_t)rb.nwin * (rb.nb + 1) * 4, s);
    k_rlc_scalars<<<grid_for(rb.cnt, 128, 1), 128, 0, s>>>(ws, d_desc, rb);
    if (ncterms) k_rlc_colsum<<<ncterms, 256, 0, s>>>(ws, rb);
    k_rlc_digits<<<(rb.N + 255) / 256, 256, 0, s>>>(d_desc, rb);
    k_rlc_scan<<<rb.nwin, 1024, 0, s>>>(rb);
    k_rlc_scatter<<<(rb.N + 255) / 256, 256, 0, s>>>(rb);
    if (ev_bucket) cudaEventRecord(ev_bucket[0], s);
    k_rlc_buckets<<<(rb.nwin * rb.nb + 127) / 128, 128, 0, s>>>(ws, d_desc, rb);
    if (ev_bucket) cudaEventRecord(ev_bucket[1], s);
    k_rlc_window_reduce<<<rb.nwin, 512, 0, s>>>(rb);
    k_rlc_final<<<1, 32, 0, s>>>(ws, d_desc, rb);
    return 8;
}
static void be_launch_verdict(const Workspace& ws, uint8_t* verdicts, be_stream s) {
    k_verdict<<<grid_for(ws.count, 256, 1), 256, 0, s>>>(ws, verdicts);
}
static void be_launch_bucket_records(const BucketArgs& a, be_stream s) { k_bucket_records<<<grid_for(a.count, BUCKET_TILE, 1), BUCKET_TILE, 0, s>>>(a); }
static void be_launch_unbucket_records(const UnbucketArgs& a, be_stream s) { k_unbucket_records<<<grid_for(a.count, BUCKET_TILE, 1), BUCKET_TILE, 0, s>>>(a); }
// entries = 2^bits multiples 1..2^bits of every constant point
static void be_launch_ctab_setup(const u32* d_enc, u32 ncp, u32* d_ctabs, u32* d_encneg, u32* d_bad, int bits, be_stream s) {
    u32 entries = 1u << bits, total = ncp * entries;
    k_ctab_setup<<<(total + 127) / 128, 128, 0, s>>>(d_enc, ncp, d_ctabs, d_encneg, d_bad, entries, bits);
}
// How many bytes of radix-2^16 constant tables an issuer may have.  README-4's 20 generators (63 MB) sit in the 126 MB L2; S16's 44
// (135 MB) do not fit entirely, but the gathers are skewed towards a few generators and the wide tables still win (570 -> 581 k/s).
#ifndef AFX_CTAB16_BUDGET_MB
#define AFX_CTAB16_BUDGET_MB 200
#endif
// AFX_CTAB16_BUDGET_MB in the environment overrides the built-in budget (0 = radix-4096 tables only).
static size_t be_ctab16_budget() {
    const char* e = std::getenv("AFX_CTAB16_BUDGET_MB");
    if (e && *e) return (size_t)std::strtoull(e, nullptr, 10) << 20;
    return (size_t)AFX_CTAB16_BUDGET_MB << 20;
}
static void be_launch_comb_setup(const u32* d_enc, u32 ncp, u32* d_comb, be_stream s) {
    u32 total = ncp * COMB_WINDOWS * COMB_ENTRIES;
    k_comb_setup<<<(total + 127) / 128, 128, 0, s>>>(d_enc, ncp, d_comb);
}
static void be_launch_link_setup(const u32* d_enc_gy, u32 ny, u32* d_out, be_stream s) { k_link_setup<<<(ny + 31) / 32, 32, 0, s>>>(d_enc_gy, ny, d_out); }
static void be_launch_primitive(u32 op, const u32* in, u32* out, u32* flags, u32 count, be_stream s) {
    k_primitive<<<(count + 127) / 128, 128, 0, s>>>(op, in, out, flags, count);
}
static void be_launch_secret_setup(const u32* d_secsc, u32 nsec, u32* d_secdig, const u32* d_Wenc, u32* d_W, u32* d_bad, be_stream s) {
    k_secret_setup<<<1, 64, 0, s>>>(d_secsc, nsec, d_secdig, d_Wenc, d_W, d_bad);
}
static void be_launch_encode(const uint8_t* data, u32* pt, uint8_t* status, u32 count, bool item_major, be_stream s) {
    k_encode<<<grid_for(count, 128, 1), 128, 0, s>>>(data, pt, status, count, item_major);
}
static void be_launch_decrypt(const u32* ct, const u32* kp, u32* tabs, uint8_t* data, u32* pt, uint8_t* status, u32 count, bool item_major, be_stream s) {
    k_decrypt<<<grid_for(count, 128, 1), 128, 0, s>>>(ct, kp, tabs, data, pt, status, count, item_major);
}
static void be_launch_keypair_scalars(const u32* ms, u32* rows, u32 count, be_stream s) {
    k_keypair_scalars<<<grid_for(count, 128, 1), 128, 0, s>>>(ms, rows, count);
}

#include "api_impl.inc"
