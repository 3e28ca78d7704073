// ssq_kernels.cu — sm_100a kernels of the alignment path and their stream-ordered launch sequence.
//
// Stage map (reference: inside `$BWA mem`, /root/reference/bin/speedseq:438; SURVEY.md §8a; measurements in DESIGN.md §5):
//   seeding  a4  default: phase-split kernels — forward walks (k_smem_fwd<1|2>, lane = read), backward sweeps (k_smem_bwd, lane = call),
//                pass-2 selection (k_smem_p2sel), greedy pass (k_smem_p3), one radix sort on (read, qb, qe) to publish the intervals.
//                Indexes with >= 2^32 rows: the per-lane state machine k_smem_m<u64> + k_smem_p3 on the 64-byte on-disk rank blocks.
//                One 256-bit load per rank query of the re-blocked 32-byte sectors.  Bound: random sector reads (L2 / HBM).
//   k_sa     a5  thread per seed occurrence, LF walk to the load-time densified SA sample.  Same bound.
//   k_chain / k_chain_coop  a6  per-lane ChainBuilder for reads with <= 16 seeds, warp per read (shared-memory chains, three
//                capacity levels) above.
//   k_ext_*  a7  seed extension in lazy rounds, jobs radix-sorted by size, one launch per query-length class; thread per
//                extension, one packed 32-bit word (H | E | query base) per column in shared memory, DPX three-way maxima.
//   k_select / k_select_heavy   resumable replay of the reference's seed-skipping rules over the candidates.
//   k_dup_* + CUB radix sort    duplicate marking (batch form, streaming set, device-pointer form used by ssq_pipe.cu / ssq_dist.cu).
// Scans and radix sorts use CUB (plumbing).  No CPU fallback exists in this library.
#include <cuda_runtime.h>
#include <cub/cub.cuh>
#include <cub/device/device_merge.cuh>
#include <mutex>
#include <condition_variable>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <vector>
#include "ssq_dev.cuh"
#include "ssq_host.h"
#include "ssq_batch.h"

#define FULL 0xffffffffu

// ------------------------------------------------------------------ warp-cooperative FM context ----
struct WarpFm {
	const DevIndex &ix;
	int lane;
	unsigned long long n_blk;
	__device__ WarpFm(const DevIndex &i, int l) : ix(i), lane(l), n_blk(0) {}
	__device__ __forceinline__ void extend(const Intv &ik, Intv ok[4], int is_back)
	{
		const u64 kf = is_back ? ik.x0 : ik.x1, ko = is_back ? ik.x1 : ik.x0;
		const u64 k = (lane & 16) ? kf - 1 + ik.x2 : kf - 1; // lower half-warp: row before the interval, upper: its last row
		const bool valid = k != (u64)-1;
		const u64 kk = k - (k >= ix.primary);
		const int l16 = lane & 15;
		u32 wv = 0, packed = 0;
		if (valid) wv = __ldg(ix.bwt + ((kk >> 7) << 4) + l16); // 16 lanes x 4 B = the 64-B block
		if (valid && l16 >= 8) {
			const int n = (int)(kk & 127) + 1 - 16 * (l16 - 8);
			if (n > 0) {
				const u32 m = n >= 16 ? 0x55555555u : (0x55555555u & ~(0xffffffffu >> (2 * n)));
				const u32 lo = wv & 0x55555555u, hi = (wv >> 1) & 0x55555555u;
				packed = __popc(~hi & ~lo & m) | __popc(~hi & lo & m) << 8 | __popc(hi & ~lo & m) << 16 | __popc(hi & lo & m) << 24;
			}
		}
		packed += __shfl_xor_sync(FULL, packed, 1);
		packed += __shfl_xor_sync(FULL, packed, 2);
		packed += __shfl_xor_sync(FULL, packed, 4); // lanes 8..15 / 24..31 now hold the per-block symbol counts
		const u32 pa = __shfl_sync(FULL, packed, 8), pb = __shfl_sync(FULL, packed, 24);
		u64 tk[4], tl[4];
#pragma unroll
		for (int c = 0; c < 4; ++c) {
			u32 alo = __shfl_sync(FULL, wv, 2 * c), ahi = __shfl_sync(FULL, wv, 2 * c + 1);
			u32 blo = __shfl_sync(FULL, wv, 16 + 2 * c), bhi = __shfl_sync(FULL, wv, 17 + 2 * c);
			tk[c] = ((u64)ahi << 32 | alo) + ((pa >> (8 * c)) & 0xff);
			tl[c] = ((u64)bhi << 32 | blo) + ((pb >> (8 * c)) & 0xff);
		}
		n_blk += 2;
		u64 nf[4], ns[4], no[4];
#pragma unroll
		for (int c = 0; c < 4; ++c) { nf[c] = ix.L2[c] + 1 + tk[c]; ns[c] = tl[c] - tk[c]; }
		no[3] = ko + (kf <= ix.primary && kf + ik.x2 - 1 >= ix.primary);
		no[2] = no[3] + ns[3]; no[1] = no[2] + ns[2]; no[0] = no[1] + ns[1];
#pragma unroll
		for (int c = 0; c < 4; ++c) {
			ok[c].x2 = ns[c];
			if (is_back) { ok[c].x0 = nf[c]; ok[c].x1 = no[c]; } else { ok[c].x1 = nf[c]; ok[c].x0 = no[c]; }
		}
	}
};

// ----------------------------------------------------------------------------- k_smem ----
// grid: persistent, blockDim = 32*warps; dynamic smem = warps * 2*(lcap+1) * sizeof(Intv)
__global__ void __launch_bounds__(256) k_smem(DevIndex ix, ssq_opts_t opt, int n_reads, const uint8_t *__restrict__ seq, const u64 *__restrict__ read_off,
                                              int lcap, Intv *scratch, int scratch_cap, Intv *pool, u64 pool_cap, unsigned long long *pool_n,
                                              u64 *intv_off, i32 *intv_cnt, i32 *l_rep_out, int *work, int *err, Counters *cnt)
{
	extern __shared__ __align__(16) unsigned char smem_raw[];
	const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, wpb = blockDim.x >> 5;
	Intv *bufA = (Intv*)smem_raw + (size_t)wib * 2 * (lcap + 1), *bufB = bufA + (lcap + 1);
	Intv *mem = scratch + (size_t)(blockIdx.x * wpb + wib) * scratch_cap;
	WarpFm fm(ix, lane);
	for (;;) {
		int r = 0;
		if (lane == 0) r = atomicAdd(work, 1);
		r = __shfl_sync(FULL, r, 0);
		if (r >= n_reads) break;
		const u64 off = read_off[r];
		const int len = (int)(read_off[r + 1] - off);
		int e = 0, n = 0;
		if (len > lcap) e = 3;
		else n = collect_intv(fm, ix, opt, len, seq + off, mem, scratch_cap, bufA, bufB, e);
		if (e) { if (lane == 0) atomicMax(err, e); n = 0; }
		// query bases covered by over-frequent seeds (frac_rep numerator)
		int b = 0, en = 0, l_rep = 0;
		for (int i = 0; i < n; ++i) {
			const Intv p = mem[i];
			if (p.x2 <= (u64)opt.max_occ) continue;
			if ((int)p.qb > en) { l_rep += en - b; b = p.qb; en = p.qe; } else en = en > (int)p.qe ? en : (int)p.qe;
		}
		l_rep += en - b;
		unsigned long long base = 0;
		if (lane == 0) base = atomicAdd(pool_n, (unsigned long long)n);
		base = __shfl_sync(FULL, base, 0);
		if (base + n > pool_cap) { if (lane == 0) atomicMax(err, 2); n = 0; }
		__syncwarp();
		for (int i = lane; i < n; i += 32) pool[base + i] = mem[i];
		if (lane == 0) { intv_off[r] = base; intv_cnt[r] = n; l_rep_out[r] = l_rep; }
		__syncwarp();
	}
	if (lane == 0 && fm.n_blk) atomicAdd(&cnt->occ_smem, fm.n_blk);
}

// thread-per-read variant: every lane runs the whole search of its own read with the scalar rank query (8 x LDG.128 per
// extension); ping-pong lists and the interval list live in per-thread global scratch (L1/L2 resident)
__global__ void __launch_bounds__(128) k_smem_t(DevIndex ix, ssq_opts_t opt, int n_reads, const uint8_t *__restrict__ seq, const u64 *__restrict__ read_off,
                                                int lcap, Intv *scratch, int scratch_cap, Intv *pool, u64 pool_cap, unsigned long long *pool_n,
                                                u64 *intv_off, i32 *intv_cnt, i32 *l_rep_out, int *work, int *err, Counters *cnt)
{
	const size_t per = (size_t)scratch_cap + 2 * (size_t)(lcap + 1) + (size_t)(scratch_cap + 7) / 8;
	Intv *mem = scratch + ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * per, *bufA = mem + scratch_cap, *bufB = bufA + (lcap + 1);
	ScalarFm fm(ix);
	for (;;) {
		const int r = atomicAdd(work, 1);
		if (r >= n_reads) break;
		const u64 off = read_off[r];
		const int len = (int)(read_off[r + 1] - off);
		int e = 0, n = 0;
		if (len > lcap) e = 3;
		else n = collect_intv(fm, ix, opt, len, seq + off, mem, scratch_cap, bufA, bufB, e);
		if (e) { atomicMax(err, e); n = 0; }
		int b = 0, en = 0, l_rep = 0;
		for (int i = 0; i < n; ++i) {
			const Intv p = mem[i];
			if (p.x2 <= (u64)opt.max_occ) continue;
			if ((int)p.qb > en) { l_rep += en - b; b = p.qb; en = p.qe; } else en = en > (int)p.qe ? en : (int)p.qe;
		}
		l_rep += en - b;
		unsigned long long base = atomicAdd(pool_n, (unsigned long long)n);
		if (base + n > pool_cap) { atomicMax(err, 2); n = 0; }
		for (int i = 0; i < n; ++i) pool[base + i] = mem[i];
		intv_off[r] = base; intv_cnt[r] = n; l_rep_out[r] = l_rep;
	}
	if (fm.n_blk) atomicAdd(&cnt->occ_smem, fm.n_blk);
}

// state-machine variant (default): a lane owns one machine and keeps pulling reads from the work counter; the only step
// all lanes of a warp take together is the rank query, whatever phase (forward / backward / pass 3) each is in.
// The ping-pong lists live in shared memory as 16-byte entries (k, l, s as u32 + query end) when the index has fewer than
// 2^32 rows, entries beyond `cap` (and every entry of larger indexes) go to the lane's global scratch lists.
template <class U> struct DevLists;
template <> struct DevLists<u64> {
	uint4 *sm; int cap, stride; Intv *g0, *g1;
	__device__ __forceinline__ Intv get(int id, int j) const
	{
		if (j < cap) { const uint4 v = sm[(size_t)(id * cap + j) * stride]; Intv r; r.x0 = v.x; r.x1 = v.y; r.x2 = v.z; r.qb = 0; r.qe = v.w; return r; }
		return (id ? g1 : g0)[j];
	}
	__device__ __forceinline__ void set(int id, int j, const Intv &v) const
	{
		if (j < cap) sm[(size_t)(id * cap + j) * stride] = make_uint4((u32)v.x0, (u32)v.x1, (u32)v.x2, v.qe);
		else (id ? g1 : g0)[j] = v;
	}
};
template <> struct DevLists<u32> { // entries are exactly the 16-byte shared-memory words; overflow entries keep the same form in global scratch
	uint4 *sm; int cap, stride; uint4 *g0, *g1;
	__device__ __forceinline__ Intv32 get(int id, int j) const
	{
		const uint4 v = j < cap ? sm[(id * cap + j) * stride] : (id ? g1 : g0)[j];
		Intv32 r; r.x0 = v.x; r.x1 = v.y; r.x2 = v.z; r.qb = 0; r.qe = v.w; return r;
	}
	__device__ __forceinline__ void set(int id, int j, const Intv32 &v) const
	{
		const uint4 w = make_uint4(v.x0, v.x1, v.x2, v.qe);
		if (j < cap) sm[(id * cap + j) * stride] = w; else (id ? g1 : g0)[j] = w;
	}
};

// Pass 3 of the seeding (the greedy sweep of seed_strategy1(): walk forward from x until the interval is small enough and long
// enough, emit it, restart right after it) needs nothing from passes 1 and 2 and has next to no state, so it runs as a kernel of
// its own in which every lane is in the same phase: ~30 lanes per instruction and 3-4x the occupancy of the full machine.  Its
// intervals go to a fixed slot range per read; k_smem_m merges them into the read's list before the final sort.
template <class U, bool TAB>
__global__ void __launch_bounds__(256) k_smem_p3(DevIndex ix, ssq_opts_t opt, int n_reads, const uint8_t *__restrict__ seq, const u64 *__restrict__ read_off,
                                                 int stride, Intv *p3, i32 *p3_cnt, int *work, Counters *cnt)
{
	ScalarFm fm(ix);
	const U max_intv = (U)opt.max_mem_intv;
	const int min_len = opt.min_seed_len;
	const uint8_t *q = 0;
	IntvT<U> ik;
	int r = -1, len = 0, x = 0, i = 0, qi = 0, qnext = 0, n_out = 0;
	u32 code = 0; // TAB: the walk's string so far (k-mer jump-start table, 32-bit rows only)
	bool have = false, ready = false, alive = true;
	ik.x0 = ik.x1 = ik.x2 = 0; ik.qb = ik.qe = 0;
	for (;;) {
		while (alive && !ready) { // (re)start a walk, or finish the read and take the next one
			if (!have) {
				r = atomicAdd(work, 1);
				if (r >= n_reads) { alive = false; break; }
				const u64 off = read_off[r];
				len = (int)(read_off[r + 1] - off); q = seq + off;
				x = (len < min_len || max_intv == 0) ? len : 0; n_out = 0; have = true;
			}
			while (x < len && q[x] > 3) ++x;
			if (x >= len) { p3_cnt[r] = n_out; have = false; continue; }
			set_intv(ix, q[x], ik);
			if (TAB) code = q[x];
			i = x + 1;
			if (i >= len) { x = len; continue; }
			qi = q[i];
			if (qi > 3) { x = i + 1; continue; }
			qnext = i + 1 < len ? (int)q[i + 1] : 4;
			ready = true;
		}
		if (__ballot_sync(FULL, alive) == 0) break;
		if (ready) {
			IntvT<U> okc;
			if (TAB) code = code << 2 | (u32)qi;
			if (TAB && i + 1 - x <= ix.kmer_k) { const Intv32 t = kmer_lookup(ix, i + 1 - x, code); okc.x0 = (U)t.x0; okc.x1 = (U)t.x1; okc.x2 = (U)t.x2; okc.qb = okc.qe = 0; }
			else extend1(fm, ik, 3 - qi, 0, okc);
			if (okc.x2 < max_intv && i - x >= min_len) {
				if (okc.x2 > 0 && n_out < stride) { Intv m = widen(okc); m.qb = (u32)x; m.qe = (u32)(i + 1); p3[(size_t)r * stride + n_out] = m; }
				if (okc.x2 > 0) ++n_out;
				x = i + 1; ready = false;
			} else {
				ik = okc; ++i;
				if (i >= len) { x = len; ready = false; }
				else { qi = qnext; if (qi > 3) { x = i + 1; ready = false; } else qnext = i + 1 < len ? (int)q[i + 1] : 4; }
			}
		}
	}
	if (fm.n_blk) { atomicAdd(&cnt->occ_smem, fm.n_blk); atomicAdd(&cnt->dbg[6], fm.n_blk); } // dbg[6]: this kernel's share of occ_smem
}

template <class U, int MINB, bool TAB>
__global__ void __launch_bounds__(128, MINB) k_smem_m(DevIndex ix, ssq_opts_t opt, int n_reads, const uint8_t *__restrict__ seq, const u64 *__restrict__ read_off,
                                                int lcap, int list_cap, int slow_batch, Intv *scratch, int scratch_cap, Intv *pool, u64 pool_cap, unsigned long long *pool_n,
                                                u64 *intv_off, i32 *intv_cnt, i32 *l_rep_out, int *work, int *err, Counters *cnt,
                                                const u32 *__restrict__ read_list, u32 *ovf_list, unsigned int *n_ovf,
                                                const Intv *__restrict__ p3, const i32 *__restrict__ p3_cnt, int p3_stride)
{
	// read_list: the reads to process (0 = all of 0..n_reads).  ovf_list: where to note a read whose intervals do not fit the
	// lane's scratch (it is redone by a second launch with a much larger scratch); 0 = that is an error.
	extern __shared__ uint4 list_smem[];
	const size_t per = (size_t)scratch_cap + 2 * (size_t)(lcap + 1) + (size_t)(scratch_cap + 7) / 8; // + 4-byte sort keys
	Intv *mem = scratch + ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * per, *bufA = mem + scratch_cap, *bufB = bufA + (lcap + 1);
	u32 *keys = (u32*)(bufB + (lcap + 1));
	DevLists<U> lists;
	lists.sm = list_smem + threadIdx.x; lists.cap = list_cap; lists.stride = blockDim.x; lists.g0 = (decltype(lists.g0))bufA; lists.g1 = (decltype(lists.g1))bufB;
	ScalarFm fm(ix);
	SmemMachineT<DevLists<U>, U, false, TAB> m; // the greedy pass is k_smem_p3's; TAB: short strings come from the k-mer jump-start table
	bool have = false, ready = false, alive = true, fin = false;
	int r = -1;
	const int batch = slow_batch > 0 ? slow_batch : 1;
	for (;;) {
		// bookkeeping up to the next rank query: every transition of the machine is short, lanes in different phases diverge only briefly
		if (have && !fin && !ready) { ready = m.advance(ix); fin = !ready; }
		const bool need_slow = alive && !ready; // read finished (to be published) or no read yet
		const unsigned slow_mask = __ballot_sync(FULL, need_slow), alive_mask = __ballot_sync(FULL, alive);
		if (alive_mask == 0) break;
		// publishing a read and fetching the next one are long, lane-serial jobs: a lane that needs them idles until `batch` lanes
		// do (or a quarter of the live lanes, or nobody can issue a query), then they run together
		const int n_slow = __popc(slow_mask), n_alive = __popc(alive_mask);
		if (need_slow && (n_slow >= batch || n_slow == n_alive || 4 * n_slow >= n_alive)) {
			if (fin) { // order the read's intervals, publish them
				if (p3 && !m.err) { // the greedy pass's intervals (k_smem_p3) join the list before the sort
					const int c3 = p3_cnt[r];
					if (c3 > p3_stride || m.n + c3 > m.mem_cap) m.err = 1;
					else for (int e = 0; e < c3; ++e) mem[m.n++] = p3[(size_t)r * p3_stride + e];
				}
				int n = m.finish(keys);
				bool redo = false;
				if (m.err) { n = 0; if (ovf_list) { ovf_list[atomicAdd(n_ovf, 1u)] = (u32)r; redo = true; } else atomicMax(err, 1); }
				int b = 0, en = 0, l_rep = 0;
				for (int i = 0; i < n; ++i) {
					const Intv p = mem[keys[i] & 0xffff];
					if (p.x2 <= (u64)opt.max_occ) continue;
					if ((int)p.qb > en) { l_rep += en - b; b = p.qb; en = p.qe; } else en = en > (int)p.qe ? en : (int)p.qe;
				}
				l_rep += en - b;
				unsigned long long base = atomicAdd(pool_n, (unsigned long long)n);
				if (base + n > pool_cap) { atomicMax(err, 2); n = 0; }
				for (int i = 0; i < n; ++i) pool[base + i] = mem[keys[i] & 0xffff];
				if (!redo) { intv_off[r] = base; intv_cnt[r] = n; l_rep_out[r] = l_rep; }
				have = false; fin = false;
			}
			while (!have) {
				r = atomicAdd(work, 1);
				if (r >= n_reads) { alive = false; break; }
				if (read_list) r = (int)read_list[r];
				const u64 off = read_off[r];
				const int len = (int)(read_off[r + 1] - off);
				if (len > lcap) { atomicMax(err, 3); intv_off[r] = 0; intv_cnt[r] = 0; l_rep_out[r] = 0; continue; }
				m.init(opt, len, seq + off, mem, scratch_cap, lists, p3 != 0);
				have = true;
			}
		}
		if (ready) { // the step all lanes that have a query take together
			IntvT<U> okc;
			if (!(TAB && m.table_hit(ix, okc))) extend1(fm, m.in, m.qc, m.is_back, okc);
			m.post(okc);
			ready = false;
		}
	}
	if (fm.n_blk) atomicAdd(&cnt->occ_smem, fm.n_blk);
}

// ------------------------------------------------------- phase-split seeding (variant 3) ----
// Every kernel here has all its lanes in ONE phase of the algorithm (what made k_smem_p3 3.8x as efficient per rank block as the
// state machine).  Data flow, all in device memory, counters in Split:
//   k_smem_fwd<1>  per read: the forward walks of pass 1, one after the other (the next starts where the previous ended)
//                  -> a SeedCall + forward list per walk
//   k_smem_bwd     per call: its backward sweeps (SmemMachineT started in its backward phase) -> intervals, tagged with the read
//   k_smem_p2sel   per pass-1 interval: long and rare enough -> a pass-2 call request (x = its middle, min_intv = its size + 1)
//   k_smem_fwd<2>  per request: the forward walk;  k_smem_bwd again for those calls
//   k_smem_p3 (+ k_smem_p3_append): the greedy pass
//   sort by (read, qb, qe) -> pool, intv_off/intv_cnt, l_rep   (equal keys are identical intervals)
struct Split { unsigned long long n_calls, n_calls1, n_fl, n_mems, n_mems1, need_calls; int err, pad; int wk[8]; }; // need_calls: n_calls before clamping to the pool size

// space for n items from a shared counter, one atomic per group of converged lanes
__device__ __forceinline__ unsigned long long group_alloc(unsigned long long *ctr, unsigned int n)
{
	const unsigned mask = __activemask();
	const int lane = threadIdx.x & 31, leader = __ffs(mask) - 1;
	unsigned int pre = 0, tot = 0;
	for (unsigned m = mask; m; m &= m - 1) { const int src = __ffs(m) - 1; const unsigned int v = __shfl_sync(mask, n, src); if (src < lane) pre += v; tot += v; }
	unsigned long long base = 0;
	if (lane == leader) base = atomicAdd(ctr, (unsigned long long)tot);
	base = __shfl_sync(mask, base, leader);
	return base + pre;
}

// PASS 1: lane = read, walks x = 0, ret, ret', ...; PASS 2: lane = call request (read, x, min_intv given), one walk
template <int PASS, bool TAB>
__global__ void __launch_bounds__(256) k_smem_fwd(DevIndex ix, ssq_opts_t opt, int n_reads, const uint8_t *__restrict__ seq, const u64 *__restrict__ read_off,
                                                  int lcap, FwdEntry *stage, SeedCall *calls, u64 call_cap, FwdEntry *fl, u64 fl_cap, Split *sp, Counters *cnt)
{
	ScalarFm fm(ix);
	FwdEntry *st = stage + ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * (size_t)(lcap + 1);
	const uint8_t *q = 0;
	Intv32 ik; ik.x0 = ik.x1 = ik.x2 = 0; ik.qb = ik.qe = 0;
	int r = -1, len = 0, x = 0, i = 0, qi = 0, qnext = 0, n_list = 0;
	u32 min_intv = 1, code = 0; // code (TAB): the walk's string so far, for the k-mer jump-start table
	unsigned long long slot = 0; // PASS 2: the request being served
	bool have = false, ready = false, alive = true;
	const unsigned long long lo2 = PASS == 2 ? sp->n_calls1 : 0, hi2 = PASS == 2 ? sp->n_calls : 0;
	auto push = [&]() { FwdEntry e; e.x0 = ik.x0; e.x1 = ik.x1; e.x2 = ik.x2; e.qe = ik.qe; st[n_list++] = e; };
	auto flush = [&]() { // the walk from x is complete: hand the call over
		const unsigned long long off = group_alloc(&sp->n_fl, (unsigned)n_list);
		unsigned long long c = slot;
		if (PASS == 1) c = group_alloc(&sp->n_calls, 1u);
		const bool fits = off + n_list <= fl_cap;
		if (!fits || c >= call_cap) atomicMax(&sp->err, 2); // a pool is too small: the host grows it and runs the stage again
		if (c < call_cap) { // the slot always gets a well-formed record; list_n == 0 tells the backward kernel to skip it
			if (fits) for (int e = 0; e < n_list; ++e) fl[off + e] = st[e];
			SeedCall sc; sc.read = (u32)r; sc.pk = SeedCall::pack(x, len, x >= 1 ? (int)q[x - 1] : 4, x >= 2 ? (int)q[x - 2] : 4);
			sc.min_intv = min_intv; sc.list_n = fits ? (u32)n_list : 0u; sc.list_off = fits ? off : 0; sc.seq_off = (u64)(q - seq);
			calls[c] = sc;
		}
		if (PASS == 1) x = (int)st[n_list - 1].qe; else have = false;
		ready = false;
	};
	for (;;) {
		while (alive && !ready) {
			if (!have) {
				if (PASS == 1) {
					r = atomicAdd(&sp->wk[0], 1);
					if (r >= n_reads) { alive = false; break; }
					const u64 off = read_off[r];
					len = (int)(read_off[r + 1] - off); q = seq + off;
					x = len < opt.min_seed_len ? len : 0;
					if (len > lcap) { atomicMax(&sp->err, 3); x = len; }
				} else {
					slot = lo2 + (unsigned long long)atomicAdd(&sp->wk[2], 1);
					if (slot >= hi2) { alive = false; break; }
					const SeedCall sc = calls[slot];
					r = (int)sc.read; x = sc.x(); min_intv = sc.min_intv;
					len = sc.len(); q = seq + sc.seq_off;
				}
				have = true;
			}
			if (PASS == 1) {
				while (x < len && q[x] > 3) ++x;
				if (x >= len) { have = false; continue; }
			}
			set_intv(ix, q[x], ik); ik.qe = (u32)(x + 1);
			if (TAB) code = q[x];
			i = x + 1; n_list = 0;
			if (i >= len) { push(); flush(); continue; }
			qi = q[i];
			if (qi > 3) { push(); flush(); continue; }
			qnext = i + 1 < len ? (int)q[i + 1] : 4;
			ready = true;
		}
		if (__ballot_sync(FULL, alive) == 0) break;
		if (ready) {
			Intv32 okc;
			if (TAB) code = code << 2 | (u32)qi;
			if (TAB && i + 1 - x <= ix.kmer_k) okc = kmer_lookup(ix, i + 1 - x, code); else extend1(fm, ik, 3 - qi, 0, okc);
			bool end = false;
			if (okc.x2 != ik.x2) { push(); end = okc.x2 < min_intv; }
			if (!end) {
				ik = okc; ik.qe = (u32)(i + 1); ++i;
				if (i >= len) { push(); end = true; }
				else { qi = qnext; if (qi > 3) { push(); end = true; } else qnext = i + 1 < len ? (int)q[i + 1] : 4; }
			}
			if (end) flush();
		}
	}
	if (fm.n_blk) atomicAdd(&cnt->occ_smem, fm.n_blk);
}

// backward sweeps of the calls [lo, hi): lane = call
template <int MINB>
__global__ void __launch_bounds__(128, MINB) k_smem_bwd(DevIndex ix, ssq_opts_t opt, const uint8_t *__restrict__ seq, const u64 *__restrict__ read_off, int lcap, int list_cap,
                                                        Intv *scratch, int scratch_cap, const SeedCall *__restrict__ calls, const FwdEntry *__restrict__ fl, int second,
                                                        Intv *mems, u32 *memr, u64 mem_cap, Split *sp, Counters *cnt)
{
	extern __shared__ uint4 list_smem[];
	const size_t per = (size_t)scratch_cap + (size_t)(lcap + 1); // output of one call + overflow of the two lists as 16-byte entries
	Intv *mem = scratch + ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * per;
	uint4 *bufA = (uint4*)(mem + scratch_cap), *bufB = bufA + (lcap + 1);
	DevLists<u32> lists;
	lists.sm = list_smem + threadIdx.x; lists.cap = list_cap; lists.stride = blockDim.x; lists.g0 = bufA; lists.g1 = bufB;
	ScalarFm fm(ix);
	SmemMachineT<DevLists<u32>, u32, false> m;
	const unsigned long long lo = second ? sp->n_calls1 : 0, hi = second ? sp->n_calls : sp->n_calls1;
	bool have = false, ready = false, alive = true;
	u32 rd = 0;
	for (;;) {
		while (alive && !ready) {
			if (have) { // call complete: its intervals go to the pool, tagged with the read
				if (m.err) atomicMax(&sp->err, 1);
				else if (m.n > 0) {
					const unsigned long long base = group_alloc(&sp->n_mems, (unsigned)m.n);
					if (base + m.n > mem_cap) atomicMax(&sp->err, 2);
					else for (int e = 0; e < m.n; ++e) { mems[base + e] = mem[e]; memr[base + e] = rd; }
				}
				have = false;
			}
			const unsigned long long c = lo + (unsigned long long)atomicAdd(&sp->wk[second ? 3 : 1], 1);
			if (c >= hi) { alive = false; break; }
			const SeedCall sc = calls[c];
			if (sc.list_n == 0) continue; // its forward list did not fit the pool (the stage is being re-run with a larger one)
			rd = sc.read;
			m.init(opt, sc.len(), seq + sc.seq_off, mem, scratch_cap, lists, 1);
			m.start_backward(sc.x(), sc.min_intv, fl + sc.list_off, (int)sc.list_n, sc.b0(), sc.b1());
			have = true;
			ready = m.advance(ix);
		}
		if (__ballot_sync(FULL, alive) == 0) break;
		if (ready) {
			Intv32 okc;
			extend1(fm, m.in, m.qc, m.is_back, okc);
			m.post(okc);
			ready = m.advance(ix);
		}
	}
	if (fm.n_blk) atomicAdd(&cnt->occ_smem, fm.n_blk);
}

// the same kernel with the lean per-lane state (BwdCallT): fewer registers -> more blocks per SM, fewer instructions per step
// (SSQ_SMEM_VARIANT=4; CPU-validated through hostsim, first GPU measurement pending)
template <int MINB, bool TAB>
__global__ void __launch_bounds__(128, MINB) k_smem_bwd2(DevIndex ix, ssq_opts_t opt, const uint8_t *__restrict__ seq, int lcap, int list_cap,
                                                         Intv *scratch, int scratch_cap, const SeedCall *__restrict__ calls, const FwdEntry *__restrict__ fl, int second,
                                                         Intv *mems, u32 *memr, u64 mem_cap, Split *sp, Counters *cnt)
{
	extern __shared__ uint4 list_smem[];
	const size_t per = (size_t)scratch_cap + (size_t)(lcap + 1);
	Intv *mem = scratch + ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * per;
	uint4 *bufA = (uint4*)(mem + scratch_cap), *bufB = bufA + (lcap + 1);
	DevLists<u32> lists;
	lists.sm = list_smem + threadIdx.x; lists.cap = list_cap; lists.stride = blockDim.x; lists.g0 = bufA; lists.g1 = bufB;
	ScalarFm fm(ix);
	BwdCallT<DevLists<u32> > m;
	m.n = 0; m.err = 0;
	const unsigned long long lo = second ? sp->n_calls1 : 0, hi = second ? sp->n_calls : sp->n_calls1;
	bool have = false, ready = false, alive = true;
	u32 rd = 0;
	for (;;) {
		while (alive && !ready) {
			if (have) { // call complete: its intervals go to the pool, tagged with the read
				if (m.err) atomicMax(&sp->err, 1);
				else if (m.n > 0) {
					const unsigned long long base = group_alloc(&sp->n_mems, (unsigned)m.n);
					if (base + m.n > mem_cap) atomicMax(&sp->err, 2);
					else for (int e = 0; e < m.n; ++e) { mems[base + e] = mem[e]; memr[base + e] = rd; }
				}
				have = false;
			}
			const unsigned long long c = lo + (unsigned long long)atomicAdd(&sp->wk[second ? 3 : 1], 1);
			if (c >= hi) { alive = false; break; }
			const SeedCall sc = calls[c];
			if (sc.list_n == 0) continue; // its forward list did not fit the pool (the stage is being re-run with a larger one)
			rd = sc.read;
			m.start(opt, sc.len(), seq + sc.seq_off, mem, scratch_cap, lists, sc.x(), sc.min_intv, fl + sc.list_off, (int)sc.list_n, sc.b0(), sc.b1());
			if (TAB) m.use_table(ix.kmer_k);
			have = true;
			ready = m.advance();
		}
		if (__ballot_sync(FULL, alive) == 0) break;
		if (ready) {
			Intv32 okc;
			if (!(TAB && m.table_hit(ix, okc))) extend1(fm, m.in, m.c, 1, okc);
			m.post(okc);
			ready = m.advance();
		}
	}
	if (fm.n_blk) atomicAdd(&cnt->occ_smem, fm.n_blk);
}

// range bookkeeping between the kernels; the counters keep counting when a pool is full, the ranges the next kernels walk must not
// copies the running rank-block counter into a diagnostic slot (brackets one kernel's share of the seeding stage's algorithmic bytes)
__global__ void k_cnt_mark(Counters *c, int slot) { c->dbg[slot] = c->occ_smem; }
__global__ void k_smem_snapshot(Split *sp, u64 call_cap, u64 mem_cap, int set1)
{
	if (sp->n_calls > sp->need_calls) sp->need_calls = sp->n_calls;
	if (sp->n_calls > call_cap) sp->n_calls = call_cap;
	if (set1) { sp->n_calls1 = sp->n_calls; sp->n_mems1 = sp->n_mems < mem_cap ? sp->n_mems : mem_cap; }
}

__global__ void k_smem_p2sel(ssq_opts_t opt, const uint8_t *__restrict__ seq, const u64 *__restrict__ read_off, const Intv *__restrict__ mems, const u32 *__restrict__ memr,
                             SeedCall *calls, u64 call_cap, Split *sp)
{
	const unsigned long long n1 = sp->n_mems1;
	const int split_len = (int)(opt.min_seed_len * opt.split_factor + .499f);
	for (unsigned long long t = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; t < n1; t += (unsigned long long)gridDim.x * blockDim.x) {
		const Intv p = mems[t];
		const int start = (int)p.qb, end = (int)p.qe;
		if (end - start < split_len || p.x2 > (u64)opt.split_width) continue;
		const unsigned long long c = group_alloc(&sp->n_calls, 1u);
		if (c >= call_cap) { atomicMax(&sp->err, 2); continue; }
		SeedCall sc; sc.read = memr[t];
		const u64 off = read_off[sc.read];
		const int x = (start + end) >> 1, len = (int)(read_off[sc.read + 1] - off);
		sc.pk = SeedCall::pack(x, len, x >= 1 ? (int)seq[off + x - 1] : 4, x >= 2 ? (int)seq[off + x - 2] : 4);
		sc.min_intv = (u32)(p.x2 + 1); sc.list_n = 0; sc.list_off = 0; sc.seq_off = off;
		calls[c] = sc;
	}
}

__global__ void k_smem_p3_append(int n_reads, const Intv *__restrict__ p3, const i32 *__restrict__ p3_cnt, int stride, Intv *mems, u32 *memr, u64 mem_cap, Split *sp)
{
	const int r = blockIdx.x * blockDim.x + threadIdx.x;
	if (r >= n_reads) return;
	const int c = p3_cnt[r];
	if (c <= 0) return;
	const unsigned long long base = group_alloc(&sp->n_mems, (unsigned)c);
	if (base + c > mem_cap || c > stride) { atomicMax(&sp->err, 2); return; }
	for (int e = 0; e < c; ++e) { mems[base + e] = p3[(size_t)r * stride + e]; memr[base + e] = (u32)r; }
}

__global__ void k_smem_keys(u64 n, const Intv *__restrict__ mems, const u32 *__restrict__ memr, u64 *keys, u32 *idx)
{
	const u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
	if (t >= n) return;
	keys[t] = (u64)memr[t] << 16 | (u64)(mems[t].qb & 0xff) << 8 | (u64)(mems[t].qe & 0xff);
	idx[t] = (u32)t;
}
__global__ void k_smem_publish(u64 n, const u64 *__restrict__ keys, const u32 *__restrict__ idx, const Intv *__restrict__ mems, Intv *pool, u64 *intv_off, i32 *intv_cnt)
{
	const u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
	if (t >= n) return;
	pool[t] = mems[idx[t]];
	const u32 r = (u32)(keys[t] >> 16);
	if (t == 0 || (u32)(keys[t - 1] >> 16) != r) intv_off[r] = t;
	atomicAdd(&intv_cnt[r], 1);
}
__global__ void k_smem_lrep(int n_reads, ssq_opts_t opt, const Intv *__restrict__ pool, const u64 *__restrict__ intv_off, const i32 *__restrict__ intv_cnt, i32 *l_rep_out)
{
	const int r = blockIdx.x * blockDim.x + threadIdx.x;
	if (r >= n_reads) return;
	const Intv *mem = pool + intv_off[r];
	int b = 0, en = 0, l_rep = 0;
	for (int i = 0; i < intv_cnt[r]; ++i) {
		const Intv p = mem[i];
		if (p.x2 <= (u64)opt.max_occ) continue;
		if ((int)p.qb > en) { l_rep += en - b; b = p.qb; en = p.qe; } else en = en > (int)p.qe ? en : (int)p.qe;
	}
	l_rep_out[r] = l_rep + (en - b);
}

// ------------------------------------------------------------------------------- k_sa ----
__global__ void k_occ_count(const Intv *__restrict__ pool, u64 n, int max_occ, u32 *nocc)
{
	u64 g = (u64)blockIdx.x * blockDim.x + threadIdx.x;
	if (g >= n) return;
	u64 step;
	nocc[g] = (u32)intv_occ_count(pool[g].x2, max_occ, step);
}

// owner[t] = the interval seed t comes from = the last g with seed_off[g] <= t: every interval drops its index at its first seed, a
// running maximum fills the rest (one coalesced pass instead of a 24-step dependent binary search per seed)
__global__ void k_sa_owner(u64 n_intv, const u64 *__restrict__ seed_off, u32 *owner)
{
	const u64 g = (u64)blockIdx.x * blockDim.x + threadIdx.x;
	if (g < n_intv && seed_off[g + 1] > seed_off[g]) owner[seed_off[g]] = (u32)g;
}

__global__ void __launch_bounds__(256) k_sa(DevIndex ix, ssq_opts_t opt, const Intv *__restrict__ pool, const u64 *__restrict__ seed_off, const u32 *__restrict__ owner,
                                            u64 n_seeds, Seed *seeds, Counters *cnt)
{
	u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
	unsigned long long n_sa = 0, n_blk = 0;
	if (t < n_seeds) {
		const u64 lo = owner[t];
		const Intv p = pool[lo];
		u64 step;
		intv_occ_count(p.x2, opt.max_occ, step);
		ScalarFm fm(ix);
		Seed s;
		s.rbeg = (i64)sa_lookup(fm, p.x0 + (t - seed_off[lo]) * step, n_sa);
		s.qbeg = (i32)p.qb; s.len = (i32)(p.qe - p.qb);
		seeds[t] = s;
		n_blk = fm.n_blk;
	}
	// one atomic per warp
	for (int o = 16; o; o >>= 1) { n_sa += __shfl_xor_sync(FULL, n_sa, o); n_blk += __shfl_xor_sync(FULL, n_blk, o); }
	if ((threadIdx.x & 31) == 0 && n_sa) { atomicAdd(&cnt->sa_reads, n_sa); atomicAdd(&cnt->occ_sa, n_blk); }
}

__global__ void k_sa_rows(DevIndex ix, u64 n, const u64 *__restrict__ rows, u64 *pos)
{
	u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
	if (t >= n) return;
	ScalarFm fm(ix);
	unsigned long long n_sa = 0;
	pos[t] = sa_lookup(fm, rows[t], n_sa);
}

// ---------------------------------------------------------------------------- k_chain ----
__global__ void __launch_bounds__(128) k_chain(DevIndex ix, ssq_opts_t opt, int n_reads, const u64 *__restrict__ read_off, const u64 *__restrict__ intv_off,
                                               const i32 *__restrict__ intv_cnt, const i32 *__restrict__ l_rep, const u64 *__restrict__ seed_off,
                                               const Seed *__restrict__ seeds, i32 *chain_of, ChainRec *ch, i32 *ord, WIdx *wi, Seed *sorted, ChainRec *outc, KeptChain *kp,
                                               i32 *n_kept, u32 *n_kseeds, int *work, Counters *cnt, const int *__restrict__ heavy_thresh_p, u32 *heavy_list, unsigned int *n_heavy)
{
	const int heavy_thresh = *heavy_thresh_p;
	unsigned long long cyc_add = 0, cyc_fin = 0, cyc_fetch = 0, max_read = 0, max_n = 0, t_read0 = 0;
	// persistent per-lane machine: the step every lane of the warp takes together is "add my read's next seed to its chains"
	ChainBuilder b;
	int r = -1, i = 0;
	u64 s0 = 0;
	bool have = false;
	for (;;) {
		bool done = false;
		while (!have || i >= b.n) {
			if (have) { // read finished: regroup, weigh, sort, filter, publish
				const long long tf0 = clock64();
				const int nk = b.finish(opt);
				cyc_fin += clock64() - tf0;
				{ const unsigned long long tr = clock64() - t_read0; if (tr > max_read) { max_read = tr; max_n = (unsigned long long)b.n << 32 | (unsigned)b.n_ch; } }
				u32 ns = 0;
				for (int c = 0; c < nk; ++c) ns += (u32)outc[s0 + c].n;
				n_kept[r] = nk; n_kseeds[r] = ns;
				have = false;
			}
			const long long tq0 = clock64();
			r = atomicAdd(work, 1);
			if (r >= n_reads) { done = true; break; }
			const int ni = intv_cnt[r];
			int n = 0;
			t_read0 = tq0;
			if (ni > 0) { s0 = seed_off[intv_off[r]]; n = (int)(seed_off[intv_off[r] + ni] - s0); }
			if (n == 0) { n_kept[r] = 0; n_kseeds[r] = 0; continue; }
			if (n > heavy_thresh) { heavy_list[atomicAdd(n_heavy, 1u)] = (u32)r; continue; } // gets a warp of its own in k_chain_coop
			b.init((int)(read_off[r + 1] - read_off[r]), n, seeds + s0, l_rep[r], chain_of + s0, ch + s0, ord + s0, wi + s0, sorted + s0, outc + s0, kp + s0);
			i = 0; have = true;
			cyc_fetch += clock64() - tq0;
		}
		if (done) break;
		{ const long long ta0 = clock64(); b.add_seed(ix, opt, i++); cyc_add += clock64() - ta0; }
	}
	atomicAdd(&cnt->dbg[0], cyc_add); atomicAdd(&cnt->dbg[1], cyc_fin); atomicAdd(&cnt->dbg[2], cyc_fetch);
	atomicMax(&cnt->dbg[3], max_read);
	if (max_read && max_read == cnt->dbg[3]) cnt->dbg[4] = max_n;
}

// Reads with many seeds (repeat families): one WARP per read.  In the thread-per-read kernel such a read's lane shares its warp with
// 31 lanes doing unrelated work and gets a fraction of the issue slots, which stretched its sequential critical path ~30x and made one
// read the duration of the whole kernel.  Here the warp cooperates and everything hot lives in shared memory:
//  * build.  A chain's key (pos = rbeg of its first seed) never changes and chains are only ever added, so the ORDER of the chains is
//    not needed while building — only the answer to mem_chain()'s look-up: "the first chain whose key equals rbeg, else the last chain
//    with a smaller key", where chains with equal keys stand as (oldest, then the others newest first).  Give every chain the
//    static 64-bit key ((pos << 13 | tie) << 13) | id with tie = 0 for the first chain of its pos and 8191 - id for later ones:
//    the reference's order is then simply ascending key, and the look-up is ONE reduction — the largest key <= ((rbeg << 26) | 8191)
//    (it is the first chain of pos == rbeg if there is one, else the last chain before it).  Each lane scans a 32-strided slice of
//    the (unsorted) key array, two REDUX instructions merge them.  No insertion shifts, no tree.  Seeds are fetched 32 at a time
//    and their contig ids computed one per lane.  (pos < 2^37, id < 8192.)
//  * finish.  Order = rank sort on that key; seed regrouping is a
//    scatter (each seed knows its rank inside its chain from the build); weights one chain per lane; the weight sort is the
//    reference's introsort (its order of equal weights matters) run by lane 0 on shared memory; the O(n^2) overlap filter tests 32
//    kept chains per step and takes the first "drop" position from a ballot.
// `cap` chains fit (48 bytes each); a read that needs more is passed on (to the same kernel launched with all of an SM's shared
// memory per warp) or, at the last level, built by lane 0 with the generic ChainBuilder.
struct CoopSmem {
	i64 *pos, *last_r; i32 *tie, *rid, *first_q, *last_q, *last_len, *cn, *first, *kept;
	WIdx *wi; KeptChain *kp; i32 *sstart, *cw;
	__device__ void carve(unsigned char *base, int cap)
	{
		pos = (i64*)base; last_r = (i64*)(base + (size_t)8 * cap); tie = (i32*)(base + (size_t)16 * cap); rid = (i32*)(base + (size_t)20 * cap);
		first_q = (i32*)(base + (size_t)24 * cap); last_q = (i32*)(base + (size_t)28 * cap); last_len = (i32*)(base + (size_t)32 * cap);
		cn = (i32*)(base + (size_t)36 * cap); first = (i32*)(base + (size_t)40 * cap); kept = (i32*)(base + (size_t)44 * cap);
		wi = (WIdx*)pos;         // after the order is known and the chain records are written out
		kp = (KeptChain*)last_r; // 16 bytes per chain over last_r + tie + rid, all dead by the time the filter starts
		sstart = tie;            // seed_start per chain, until the filter
		cw = cn;                 // chain weight replaces the seed count once the count is in the chain record
	}
};

__global__ void __launch_bounds__(32) k_chain_coop(DevIndex ix, ssq_opts_t opt, int cap, const u64 *__restrict__ read_off, const u64 *__restrict__ intv_off,
                                                   const i32 *__restrict__ intv_cnt, const i32 *__restrict__ l_rep, const u64 *__restrict__ seed_off,
                                                   const Seed *__restrict__ seeds_, i32 *chain_of_, ChainRec *ch_, i32 *ord_, WIdx *wi_, Seed *sorted_, ChainRec *outc_, KeptChain *kp_,
                                                   i32 *n_kept, u32 *n_kseeds, int *work, const u32 *__restrict__ list, const unsigned int *__restrict__ n_list,
                                                   u32 *next_list, unsigned int *n_next)
{
	extern __shared__ __align__(16) unsigned char coop_smem[];
	CoopSmem S; S.carve(coop_smem, cap);
	const int lane = threadIdx.x;
	const unsigned int nl = *n_list;
	const i64 l_pac = ix.l_pac;
	for (;;) {
		int w = 0;
		if (lane == 0) w = atomicAdd(work, 1);
		w = __shfl_sync(FULL, w, 0);
		if ((unsigned)w >= nl) break;
		const int r = (int)list[w];
		const u64 s0 = seed_off[intv_off[r]];
		const int n = (int)(seed_off[intv_off[r] + intv_cnt[r]] - s0), len = (int)(read_off[r + 1] - read_off[r]);
		const Seed *seeds = seeds_ + s0; i32 *chain_of = chain_of_ + s0; ChainRec *ch = ch_ + s0; i32 *ord = ord_ + s0; i32 *rank_in = (i32*)(wi_ + s0);
		Seed *sorted = sorted_ + s0; ChainRec *outc = outc_ + s0;
		int n_ch = 0, nk = 0;
		u32 ns = 0;
		bool overflow = false;
		// ------------------------------------------------------------------ build ----
		for (int i0 = 0; i0 < n && !overflow; i0 += 32) {
			Seed my; my.rbeg = 0; my.qbeg = 0; my.len = 0;
			int myrid = -1;
			if (i0 + lane < n) { my = seeds[i0 + lane]; myrid = intv2rid(ix, my.rbeg, my.rbeg + my.len); }
			const int cnt = n - i0 < 32 ? n - i0 : 32;
			int my_chain = -1, my_rank = 0; // results for the seed this lane fetched
			for (int j = 0; j < cnt; ++j) {
				const i64 rbeg = __shfl_sync(FULL, my.rbeg, j);
				const int qbeg = __shfl_sync(FULL, my.qbeg, j), slen = __shfl_sync(FULL, my.len, j), rid = __shfl_sync(FULL, myrid, j);
				if (rid < 0) continue;
				// look-up over the unsorted keys: max key <= limit
				const i64 limit = (rbeg << 26) | 8191;
				i64 best = -1;
				for (int q = lane; q < n_ch; q += 32) { const i64 kq = S.pos[q]; if (kq <= limit && kq > best) best = kq; }
				{
					const int hi = (int)(best >> 32); // -1 when the lane found nothing
					const int ghi = __reduce_max_sync(FULL, hi);
					const unsigned glo = __reduce_max_sync(FULL, hi == ghi ? (unsigned)best : 0u);
					best = ghi < 0 ? -1 : ((i64)ghi << 32 | glo);
				}
				const bool exact = best >= 0 && (best >> 13) == (rbeg << 13);
				const int slot = best < 0 ? -1 : (int)(best & 8191);
				int res_chain = -1, res_rank = 0;
				bool merged = false;
				if (slot >= 0) { // every lane evaluates the merge test on the same shared-memory words
					const i64 c_first_r = S.pos[slot] >> 26, c_last_r = S.last_r[slot];
					const int c_first_q = S.first_q[slot], c_last_q = S.last_q[slot], c_last_len = S.last_len[slot];
					const i64 qend = c_last_q + c_last_len, rend = c_last_r + c_last_len;
					if (rid == S.rid[slot]) {
						if (qbeg >= c_first_q && qbeg + slen <= qend && rbeg >= c_first_r && rbeg + slen <= rend) merged = true; // contained
						else if (!((c_last_r < l_pac || c_first_r < l_pac) && rbeg >= l_pac)) {
							const i64 x = qbeg - c_last_q, y = rbeg - c_last_r;
							if (y >= 0 && x - y <= opt.w && y - x <= opt.w && x - c_last_len < opt.max_chain_gap && y - c_last_len < opt.max_chain_gap) {
								res_chain = slot; res_rank = S.cn[slot];
								__syncwarp();
								if (lane == 0) { S.last_q[slot] = qbeg; S.last_r[slot] = rbeg; S.last_len[slot] = slen; S.cn[slot] = res_rank + 1; }
								merged = true;
							}
						}
					}
				}
				if (!merged) {
					if (n_ch >= cap) { overflow = true; break; }
					if (lane == 0) {
						S.pos[n_ch] = ((rbeg << 13 | (exact ? 8191 - n_ch : 0)) << 13) | n_ch;
						S.last_r[n_ch] = rbeg; S.first_q[n_ch] = qbeg; S.last_q[n_ch] = qbeg; S.last_len[n_ch] = slen;
						S.rid[n_ch] = rid; S.cn[n_ch] = 1;
					}
					res_chain = n_ch; res_rank = 0;
					++n_ch;
				}
				__syncwarp();
				if (lane == j) { my_chain = res_chain; my_rank = res_rank; }
			}
			if (!overflow && i0 + lane < n) { chain_of[i0 + lane] = my_chain; rank_in[i0 + lane] = my_rank; }
		}
		__syncwarp();
		if (overflow) {
			if (next_list) { if (lane == 0) next_list[atomicAdd(n_next, 1u)] = (u32)r; continue; } // retried with more shared memory
			if (lane == 0) { // last level: the generic builder
				ChainBuilder b;
				b.init(len, n, seeds, l_rep[r], chain_of, ch, ord, wi_ + s0, sorted, outc, kp_ + s0);
				for (int i = 0; i < n; ++i) b.add_seed(ix, opt, i);
				nk = b.finish(opt);
				for (int c = 0; c < nk; ++c) ns += (u32)outc[c].n;
				n_kept[r] = nk; n_kseeds[r] = ns;
			}
			__syncwarp();
			continue;
		}
		if (n_ch > 0) {
			// ----------------------------------------------------------- order ----
			for (int q = lane; q < n_ch; q += 32) {
				const i64 kq = S.pos[q];
				int rk = 0;
				for (int j = 0; j < n_ch; ++j) rk += S.pos[j] < kq;
				ord[rk] = q;
			}
			__syncwarp();
			// seed_start = exclusive scan of the seed counts in that order
			for (int base = 0, run = 0; base < n_ch; base += 32) {
				const int q = base + lane;
				const int id = q < n_ch ? ord[q] : -1;
				const int v = id >= 0 ? S.cn[id] : 0;
				int inc = v;
#pragma unroll
				for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(FULL, inc, o); if (lane >= o) inc += t; }
				if (id >= 0) S.sstart[id] = run + inc - v;
				run += __shfl_sync(FULL, inc, 31);
			}
			__syncwarp();
			const float frac_rep = (float)l_rep[r] / len;
			for (int q = lane; q < n_ch; q += 32) { // the chain records
				ChainRec c;
				c.pos = S.pos[q] >> 26; c.first_r = c.pos; c.last_r = S.last_r[q]; c.first_q = S.first_q[q]; c.last_q = S.last_q[q]; c.last_len = S.last_len[q];
				c.rid = S.rid[q]; c.n = S.cn[q]; c.w = 0; c.first = -1; c.kept = 0; c.seed_start = S.sstart[q]; c.frac_rep = frac_rep;
				ch[q] = c;
			}
			for (int i = lane; i < n; i += 32) { const int co = chain_of[i]; if (co >= 0) sorted[S.sstart[co] + rank_in[i]] = seeds[i]; }
			__syncwarp();
			// ---------------------------------------------------------- weights ----
			for (int q = lane; q < n_ch; q += 32) {
				const Seed *sd = sorted + S.sstart[q];
				const int cnq = S.cn[q];
				i64 end; int j, w2 = 0, tmp;
				for (j = 0, end = 0; j < cnq; ++j) {
					const i64 qb = sd[j].qbeg, l = sd[j].len;
					if (qb >= end) w2 += (int)l; else if (qb + l > end) w2 += (int)(qb + l - end);
					end = end > qb + l ? end : qb + l;
				}
				tmp = w2; w2 = 0;
				for (j = 0, end = 0; j < cnq; ++j) {
					const i64 rb = sd[j].rbeg, l = sd[j].len;
					if (rb >= end) w2 += (int)l; else if (rb + l > end) w2 += (int)(rb + l - end);
					end = end > rb + l ? end : rb + l;
				}
				w2 = w2 < tmp ? w2 : tmp;
				w2 = w2 < 1 << 30 ? w2 : (1 << 30) - 1;
				S.cw[q] = w2; // only this lane reads cn[q]
				ch[q].w = w2;
			}
			__syncwarp();
			for (int q = lane; q < n_ch; q += 32) { const int id = ord[q]; WIdx x; x.w = S.cw[id]; x.idx = id; S.wi[q] = x; S.first[q] = -1; S.kept[q] = 0; } // pos[] is dead
			__syncwarp();
			if (lane == 0) ks_introsort((long)n_ch, S.wi, WIdxLt());
			__syncwarp();
			// ----------------------------------------------------------- filter ----
			int n_keptc = 1;
			if (lane == 0) {
				const int id = S.wi[0].idx;
				KeptChain k0; k0.b = S.first_q[id]; k0.e = S.last_q[id] + S.last_len[id]; k0.w = S.cw[id]; k0.i = 0;
				S.kp[0] = k0; S.kept[0] = 3;
			}
			__syncwarp();
			for (int i = 1; i < n_ch; ++i) {
				const int id = S.wi[i].idx;
				const int bi = S.first_q[id], ei = S.last_q[id] + S.last_len[id], wv = S.cw[id];
				int large = 0; bool dropped = false;
				for (int base = 0; base < n_keptc && !dropped; base += 32) {
					const int kk = base + lane;
					bool ov = false, brk = false; int kji = 0;
					if (kk < n_keptc) {
						const KeptChain kj = S.kp[kk];
						kji = kj.i;
						const int b_max = kj.b > bi ? kj.b : bi, e_min = kj.e < ei ? kj.e : ei;
						if (e_min > b_max) {
							const int li = ei - bi, lj = kj.e - kj.b, min_l = li < lj ? li : lj;
							if (e_min - b_max >= min_l * opt.mask_level && min_l < opt.max_chain_gap) {
								ov = true;
								brk = wv < kj.w * opt.drop_ratio && kj.w - wv >= opt.min_seed_len << 1;
							}
						}
					}
					const unsigned m_ov = __ballot_sync(FULL, ov), m_brk = __ballot_sync(FULL, brk);
					const unsigned upto = m_brk ? (0xffffffffu >> (32 - __ffs(m_brk))) : 0xffffffffu; // lanes up to and including the first drop
					const unsigned eff = m_ov & upto;
					if (eff) large = 1;
					if ((eff >> lane & 1) && S.first[kji] < 0) S.first[kji] = i;
					if (m_brk) dropped = true;
				}
				__syncwarp();
				if (!dropped) {
					if (lane == 0) { KeptChain kn; kn.b = bi; kn.e = ei; kn.w = wv; kn.i = i; S.kp[n_keptc] = kn; S.kept[i] = large ? 2 : 3; }
					++n_keptc;
					__syncwarp();
				}
			}
			for (int q = lane; q < n_keptc; q += 32) { const int f = S.first[S.kp[q].i]; if (f >= 0) S.kept[f] = 1; }
			__syncwarp();
			if (lane == 0) {
				int i2, k2;
				for (i2 = k2 = 0; i2 < n_ch; ++i2) {
					const int kept = S.kept[i2];
					if (kept == 0 || kept == 3) continue;
					if (++k2 >= opt.max_chain_extend) break;
				}
				for (; i2 < n_ch; ++i2) if (S.kept[i2] < 3) S.kept[i2] = 0;
			}
			__syncwarp();
			// kept chains out, in weight order
			for (int base = 0; base < n_ch; base += 32) {
				const int q = base + lane;
				const bool f = q < n_ch && S.kept[q] != 0;
				const unsigned m = __ballot_sync(FULL, f);
				if (f) {
					ChainRec c = ch[S.wi[q].idx];
					c.kept = S.kept[q]; c.first = S.first[q];
					outc[nk + __popc(m & ((1u << lane) - 1))] = c;
					ns += (u32)c.n;
				}
				nk += __popc(m);
			}
#pragma unroll
			for (int o = 16; o; o >>= 1) ns += __shfl_xor_sync(FULL, ns, o);
		}
		if (lane == 0) { n_kept[r] = nk; n_kseeds[r] = ns; }
		__syncwarp();
	}
}

// --------------------------------------------------------------------------- k_extend ----
struct Task { i32 read, chain, seed; };

__global__ void k_tasks(int n_reads, const u64 *__restrict__ intv_off, const i32 *__restrict__ intv_cnt, const u64 *__restrict__ seed_off,
                        const ChainRec *__restrict__ outc, const i32 *__restrict__ n_kept, const u64 *__restrict__ task_off, Task *tasks)
{
	int r = blockIdx.x * blockDim.x + threadIdx.x;
	if (r >= n_reads || n_kept[r] == 0) return;
	const u64 s0 = seed_off[intv_off[r]];
	u64 t = task_off[r];
	for (int c = 0; c < n_kept[r]; ++c)
		for (int s = 0; s < outc[s0 + c].n; ++s) { Task k; k.read = r; k.chain = c; k.seed = s; tasks[t++] = k; }
}

// ---- seed extension as size-sorted passes -------------------------------------------------------------------
// per task: geometry (ExtInfo), left/right results, band flags.  Jobs of one direction are radix-sorted by
// (qlen << 16 | tlen) and launched per query-length class, so the lanes of a warp run near-identical DP loops and the
// shared-memory row (packed int16 H|E, word j*blockDim + lane) is sized for the class, not for the longest read.
#define EXT_NO_JOB 0xffffffffu
__device__ __forceinline__ u32 ext_key(int qlen, int tlen) { return qlen > 0 ? ((u32)qlen << 16 | (u32)(tlen < 65535 ? tlen : 65535)) : EXT_NO_JOB; }

__global__ void __launch_bounds__(256) k_ext_prep(DevIndex ix, ssq_opts_t opt, u64 n_tasks, const Task *__restrict__ tasks, const u64 *__restrict__ read_off,
                                                  const u64 *__restrict__ intv_off, const u64 *__restrict__ seed_off, const ChainRec *__restrict__ outc,
                                                  const Seed *__restrict__ sorted, ExtInfo *info)
{
	u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
	if (t >= n_tasks) return;
	const Task k = tasks[t];
	const u64 s0 = seed_off[intv_off[k.read]];
	const ChainRec c = outc[s0 + k.chain];
	ExtInfo e;
	ext_prep(ix, opt, (int)(read_off[k.read + 1] - read_off[k.read]), c, sorted + s0 + c.seed_start, k.seed, e);
	info[t] = e;
}

// jobs of this round: tasks requested (need) and not yet extended (have)
__global__ void __launch_bounds__(256) k_ext_keys(int dir, u64 n_tasks, const ExtInfo *__restrict__ info, const uint8_t *__restrict__ need, const uint8_t *__restrict__ have, u32 *key, u32 *idx)
{
	u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
	if (t >= n_tasks) return;
	u32 kk = EXT_NO_JOB;
	if (need[t] && !have[t]) { const ExtInfo e = info[t]; kk = dir == 0 ? ext_key(ext_left_qlen(e), ext_left_tlen(e)) : ext_key(ext_right_qlen(e), ext_right_tlen(e)); }
	key[t] = kk; idx[t] = (u32)t;
}

// round 0 asks for the longest seed of every kept chain (the first one mem_chain2aln() looks at)
__global__ void k_need_first(int n_reads, const u64 *__restrict__ intv_off, const u64 *__restrict__ seed_off, const ChainRec *__restrict__ outc, const Seed *__restrict__ sorted,
                             const i32 *__restrict__ n_kept, const u64 *__restrict__ task_off, uint8_t *need)
{
	int r = blockIdx.x * blockDim.x + threadIdx.x;
	if (r >= n_reads || n_kept[r] == 0) return;
	const u64 s0 = seed_off[intv_off[r]];
	u64 t = task_off[r];
	for (int c = 0; c < n_kept[r]; ++c) {
		const ChainRec ch = outc[s0 + c];
		const Seed *cs = sorted + s0 + ch.seed_start;
		int best = 0;
		for (int i = 1; i < ch.n; ++i) if (cs[i].len >= cs[best].len) best = i; // largest (len, index)
		need[t + best] = 1;
		t += ch.n;
	}
}

// bounds[c] = first sorted job whose qlen exceeds caps[c-1]; bounds[0] = 0, bounds[6] = number of real jobs
__global__ void k_ext_bounds(u64 n, const u32 *__restrict__ keys, u32 *bounds)
{
	const int caps[6] = {32, 64, 96, 128, 160, 255};
	const int c = threadIdx.x;
	if (c > 6) return;
	if (c == 0) { bounds[0] = 0; return; }
	const u32 lim = (u32)(caps[c - 1] + 1) << 16;
	u64 lo = 0, hi = n;
	while (lo < hi) { u64 mid = (lo + hi) >> 1; if (keys[mid] < lim) lo = mid + 1; else hi = mid; }
	bounds[c] = (u32)lo;
}

template <int DIR>
__global__ void __launch_bounds__(128) k_ext_run(DevIndex ix, ssq_opts_t opt, u32 job_lo, u32 job_hi, const u32 *__restrict__ order, const Task *__restrict__ tasks,
                                                 const uint8_t *__restrict__ seq, const u64 *__restrict__ read_off, const ExtInfo *__restrict__ info,
                                                 const RegCand *__restrict__ cand, ExtRes *res, u32 *retry, unsigned int *n_retry, Counters *cnt)
{
	extern __shared__ u32 eh_smem[];
	const u32 job = job_lo + blockIdx.x * blockDim.x + threadIdx.x;
	unsigned long long cells = 0, calls = 0, bytes = 0;
	if (job < job_hi) {
		const u32 t = order[job];
		const ExtInfo e = info[t];
		const uint8_t *query = seq + read_off[tasks[t].read];
		EhAcc eh; eh.base = eh_smem + threadIdx.x; eh.stride = blockDim.x;
		ExtRes r;
		if (DIR == 0) { ext_left_run(ix, opt, query, e, opt.w, eh, r, cells); bytes = (unsigned long long)e.qbeg + (ext_left_tlen(e) + 3) / 4 + 24; }
		else { ext_right_run(ix, opt, query, e, cand[t].score, opt.w, eh, r, cells); bytes = (unsigned long long)ext_right_qlen(e) + (ext_right_tlen(e) + 3) / 4 + 24; }
		calls = 1;
		res[t] = r;
		if (ext_needs_retry(opt, r)) retry[atomicAdd(n_retry, 1u)] = t;
	}
	for (int o = 16; o; o >>= 1) { cells += __shfl_xor_sync(FULL, cells, o); calls += __shfl_xor_sync(FULL, calls, o); bytes += __shfl_xor_sync(FULL, bytes, o); }
	if ((threadIdx.x & 31) == 0 && calls) { atomicAdd(&cnt->sw_calls, calls); atomicAdd(&cnt->sw_cells, cells); atomicAdd(&cnt->sw_bytes, bytes); }
}

// the rare second try with the doubled band; shared memory sized for the longest read
template <int DIR>
__global__ void __launch_bounds__(64) k_ext_retry(DevIndex ix, ssq_opts_t opt, const u32 *__restrict__ retry, const unsigned int *__restrict__ n_retry,
                                                  const Task *__restrict__ tasks, const uint8_t *__restrict__ seq, const u64 *__restrict__ read_off,
                                                  const ExtInfo *__restrict__ info, const RegCand *__restrict__ cand, ExtRes *res, uint8_t *wide, Counters *cnt)
{
	extern __shared__ u32 eh_smem[];
	const unsigned int n = *n_retry;
	unsigned long long cells = 0, calls = 0, bytes = 0;
	EhAcc eh; eh.base = eh_smem + threadIdx.x; eh.stride = blockDim.x;
	for (unsigned int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
		const u32 t = retry[i];
		const ExtInfo e = info[t];
		const uint8_t *query = seq + read_off[tasks[t].read];
		ExtRes r;
		if (DIR == 0) { ext_left_run(ix, opt, query, e, opt.w << 1, eh, r, cells); bytes += (unsigned long long)e.qbeg + (ext_left_tlen(e) + 3) / 4 + 24; }
		else { ext_right_run(ix, opt, query, e, cand[t].score, opt.w << 1, eh, r, cells); bytes += (unsigned long long)ext_right_qlen(e) + (ext_right_tlen(e) + 3) / 4 + 24; }
		++calls;
		res[t] = r;
		wide[t] = 1;
	}
	if (calls) { atomicAdd(&cnt->sw_calls, calls); atomicAdd(&cnt->sw_cells, cells); atomicAdd(&cnt->sw_bytes, bytes); }
}

__global__ void __launch_bounds__(256) k_ext_left_fin(ssq_opts_t opt, u64 n_tasks, const ExtInfo *__restrict__ info, const ExtRes *__restrict__ lres, RegCand *cand,
                                                      const uint8_t *__restrict__ need, const uint8_t *__restrict__ have)
{
	u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
	if (t >= n_tasks || !need[t] || have[t]) return;
	const ExtInfo e = info[t];
	RegCand a;
	a.qe = 0; a.re = 0; a.w = 0; a.seedcov = 0; a.seedlen0 = 0; a.frac_rep = 0.f;
	ext_left_fin(opt, e, ext_left_qlen(e) > 0, lres[t], a);
	cand[t] = a;
}

__global__ void __launch_bounds__(256) k_ext_right_fin(ssq_opts_t opt, u64 n_tasks, const Task *__restrict__ tasks, const u64 *__restrict__ intv_off,
                                                       const u64 *__restrict__ seed_off, const ChainRec *__restrict__ outc, const Seed *__restrict__ sorted,
                                                       const ExtInfo *__restrict__ info, const ExtRes *__restrict__ rres, const uint8_t *__restrict__ wide_l,
                                                       const uint8_t *__restrict__ wide_r, RegCand *cand, const uint8_t *__restrict__ need, uint8_t *have)
{
	u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
	if (t >= n_tasks || !need[t] || have[t]) return;
	const Task k = tasks[t];
	const u64 s0 = seed_off[intv_off[k.read]];
	const ChainRec c = outc[s0 + k.chain];
	const ExtInfo e = info[t];
	RegCand a = cand[t];
	ext_right_fin(opt, e, ext_right_qlen(e) > 0, rres[t], opt.w << wide_l[t], opt.w << wide_r[t], c, sorted + s0 + c.seed_start, a);
	cand[t] = a;
	have[t] = 1;
}

// batch form of ksw_extend2 on explicit byte sequences (C-ABI ssq_sw_extend_batch)
__global__ void __launch_bounds__(64) k_sw_tasks(ssq_opts_t opt, u64 n, const ssq_sw_task_t *__restrict__ tk, const uint8_t *__restrict__ qbuf,
                                                 const uint8_t *__restrict__ tbuf, ssq_sw_result_t *out)
{
	extern __shared__ u32 eh_smem[];
	u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
	if (t >= n) return;
	const ssq_sw_task_t k = tk[t];
	const uint8_t *q = qbuf + k.q_off, *tg = tbuf + k.t_off;
	EhAcc eh; eh.base = eh_smem + threadIdx.x; eh.stride = blockDim.x;
	ssq_sw_result_t r;
	unsigned long long cells = 0;
	r.score = sw_extend(opt, k.qlen, [&](int j) { return (int)q[j]; }, k.tlen, [&](int i) { return (int)tg[i]; }, k.w, k.end_bonus, k.zdrop, k.h0, eh,
	                    r.qle, r.tle, r.gtle, r.gscore, r.max_off, cells);
	out[t] = r;
}

// --------------------------------------------------------------------------- k_select ----
// mem_chain2aln()'s seed loop per read over the candidates computed so far.  A read whose walk reaches a seed that must be
// extended but has no candidate yet flags that seed (need), records where it stopped (SelState) and goes on the next round's
// list; the host runs another extension round for the flagged seeds and the walk RESUMES at that seed.  force_all: flag every
// remaining seed of an unfinished read at once (bounds the number of rounds).  list_in == 0: all reads (first round).
__global__ void __launch_bounds__(128) k_select(ssq_opts_t opt, int n_in, const u32 *__restrict__ list_in, const u64 *__restrict__ read_off, const u64 *__restrict__ intv_off,
                                                const u64 *__restrict__ seed_off, const ChainRec *__restrict__ outc, const Seed *__restrict__ sorted,
                                                const i32 *__restrict__ n_kept, const u64 *__restrict__ task_off, const RegCand *__restrict__ cand, u64 *srt,
                                                RegCand *regs, u32 *n_regs, const uint8_t *__restrict__ have, uint8_t *need, SelState *state, int force_all,
                                                u32 *list_out, unsigned int *n_unfinished, int *work, const int *__restrict__ heavy_thresh, u32 *heavy_list, unsigned int *n_heavy)
{
	const int thresh = *heavy_thresh;
	for (;;) {
		const int w = atomicAdd(work, 1);
		if (w >= n_in) return;
		const int r = list_in ? (int)list_in[w] : w;
		const u64 t0 = task_off[r];
		if ((int)(task_off[r + 1] - t0) > thresh) { heavy_list[atomicAdd(n_heavy, 1u)] = (u32)r; continue; } // taken by a warp of its own
		const u64 s0 = seed_off[intv_off[r]];
		SelState st = state[r];
		const bool complete = select_read(opt, (int)(read_off[r + 1] - read_off[r]), n_kept[r], outc + s0, sorted + s0, cand + t0, srt + t0, regs + t0, have + t0, need + t0, force_all, st);
		if (complete) n_regs[r] = (u32)st.n_out;
		else { state[r] = st; list_out[atomicAdd(n_unfinished, 1u)] = (u32)r; }
	}
}

// The same walk with the warp's 32 lanes sharing one chain: the seed order comes from a rank sort (keys are unique, so any sort
// gives the reference's order), and the two inner tests — "is this seed inside an accepted region" and "does a longer seed
// overlap it off-diagonal" — only ask whether SOME element satisfies a predicate, so 32 elements are tested per step.
__device__ int select_regions_warp(const ssq_opts_t &opt, int l_query, const ChainRec &c, const Seed *cs, const RegCand *cand, u64 *srt, u64 *tmp,
                                   RegCand *out, int &n_out, const uint8_t *have, int resume_k, int &stop_k, int lane)
{
	int k;
	if (resume_k >= 0) {
		k = resume_k;
		const u32 si = (u32)srt[k];
		if (!have[si]) { stop_k = k; return (int)si; }
		if (lane == 0) out[n_out] = cand[si];
		++n_out; --k;
		__syncwarp();
	} else {
		for (int i = lane; i < c.n; i += 32) tmp[i] = (u64)(u32)cs[i].len << 32 | (u32)i; // seed score == len
		__syncwarp();
		for (int i = lane; i < c.n; i += 32) {
			const u64 key = tmp[i];
			int rank = 0;
			for (int j = 0; j < c.n; ++j) rank += tmp[j] < key;
			srt[rank] = key;
		}
		__syncwarp();
		k = c.n - 1;
	}
	for (; k >= 0; --k) {
		const u32 si = (u32)srt[k];
		const Seed s = cs[si];
		bool inside = false;
		for (int base = 0; base < n_out && !inside; base += 32) {
			const int i = base + lane;
			bool h = false;
			if (i < n_out) {
				const RegCand &p = out[i];
				if (!(s.rbeg < p.rb || s.rbeg + s.len > p.re || s.qbeg < p.qb || s.qbeg + s.len > p.qe) && !(s.len - p.seedlen0 > .1 * l_query)) {
					i64 rd; int qd, w, max_gap;
					qd = s.qbeg - p.qb; rd = s.rbeg - p.rb;
					max_gap = cal_max_gap(opt, qd < rd ? qd : (int)rd);
					w = max_gap < p.w ? max_gap : p.w;
					if (qd - rd < w && rd - qd < w) h = true;
					else {
						qd = p.qe - (s.qbeg + s.len); rd = p.re - (s.rbeg + s.len);
						max_gap = cal_max_gap(opt, qd < rd ? qd : (int)rd);
						w = max_gap < p.w ? max_gap : p.w;
						if (qd - rd < w && rd - qd < w) h = true;
					}
				}
			}
			inside = __any_sync(FULL, h);
		}
		if (inside) {
			bool overlap = false;
			for (int base = k + 1; base < c.n && !overlap; base += 32) {
				const int i = base + lane;
				bool h = false;
				if (i < c.n && srt[i] != 0) {
					const Seed t = cs[(u32)srt[i]];
					if (!(t.len < s.len * .95)) {
						if (s.qbeg <= t.qbeg && s.qbeg + s.len - t.qbeg >= s.len >> 2 && t.qbeg - s.qbeg != t.rbeg - s.rbeg) h = true;
						else if (t.qbeg <= s.qbeg && t.qbeg + t.len - s.qbeg >= s.len >> 2 && s.qbeg - t.qbeg != s.rbeg - t.rbeg) h = true;
					}
				}
				overlap = __any_sync(FULL, h);
			}
			if (!overlap) { __syncwarp(); if (lane == 0) srt[k] = 0; __syncwarp(); continue; }
		}
		if (!have[si]) { stop_k = k; return (int)si; }
		if (lane == 0) out[n_out] = cand[si];
		++n_out;
		__syncwarp();
	}
	return -1;
}

__global__ void __launch_bounds__(128) k_select_heavy(ssq_opts_t opt, const u64 *__restrict__ read_off, const u64 *__restrict__ intv_off,
                                                      const u64 *__restrict__ seed_off, const ChainRec *__restrict__ outc_, const Seed *__restrict__ sorted_,
                                                      const i32 *__restrict__ n_kept, const u64 *__restrict__ task_off, const RegCand *__restrict__ cand, u64 *srt, u64 *tmp,
                                                      RegCand *regs, u32 *n_regs, const uint8_t *__restrict__ have, uint8_t *need, SelState *state, int force_all,
                                                      u32 *list_out, unsigned int *n_unfinished, int *work, const u32 *__restrict__ heavy_list, const unsigned int *__restrict__ n_heavy)
{
	const int lane = threadIdx.x & 31;
	const unsigned int nh = *n_heavy;
	for (;;) {
		int w = 0;
		if (lane == 0) w = atomicAdd(work, 1);
		w = __shfl_sync(FULL, w, 0);
		if ((unsigned)w >= nh) break;
		const int r = (int)heavy_list[w];
		const u64 t0 = task_off[r], s0 = seed_off[intv_off[r]];
		const int len = (int)(read_off[r + 1] - read_off[r]), nk = n_kept[r];
		const ChainRec *outc = outc_ + s0; const Seed *sorted = sorted_ + s0;
		const SelState st = state[r];
		int c = st.c, n_out = st.n_out, kk = st.kp1 - 1;
		u32 t = st.t_rel;
		bool complete = true;
		for (; c < nk; ++c, kk = -1) {
			const ChainRec ch = outc[c];
			int stop_k = -1;
			const int miss = select_regions_warp(opt, len, ch, sorted + ch.seed_start, cand + t0 + t, srt + t0 + t, tmp + t0 + t, regs + t0, n_out, have + t0 + t, kk, stop_k, lane);
			if (miss >= 0) {
				if (force_all) { u32 e = t; for (int cc = c; cc < nk; ++cc) e += (u32)outc[cc].n; for (u32 x = t + lane; x < e; x += 32) need[t0 + x] = 1; }
				else if (lane == 0) need[t0 + t + miss] = 1;
				if (lane == 0) { SelState o; o.c = c; o.n_out = n_out; o.kp1 = stop_k + 1; o.t_rel = t; state[r] = o; list_out[atomicAdd(n_unfinished, 1u)] = (u32)r; }
				complete = false;
				break;
			}
			t += (u32)ch.n;
		}
		if (complete && lane == 0) n_regs[r] = (u32)n_out;
		__syncwarp();
	}
}

__global__ void k_gather_regs(int n_reads, const u64 *__restrict__ task_off, const u64 *__restrict__ reg_off, const u32 *__restrict__ n_regs,
                              const RegCand *__restrict__ regs, ssq_alnreg_t *out)
{
	int r = blockIdx.x * blockDim.x + threadIdx.x;
	if (r >= n_reads) return;
	for (u32 i = 0; i < n_regs[r]; ++i) {
		const RegCand a = regs[task_off[r] + i];
		ssq_alnreg_t o;
		o.rb = a.rb; o.re = a.re; o.qb = a.qb; o.qe = a.qe; o.rid = a.rid; o.score = a.score; o.truesc = a.truesc; o.w = a.w;
		o.seedcov = a.seedcov; o.seedlen0 = a.seedlen0; o.frac_rep = a.frac_rep; o.read_id = r;
		out[reg_off[r] + i] = o;
	}
}

__global__ void k_gather_intv(int n_reads, const u64 *__restrict__ intv_off, const i32 *__restrict__ intv_cnt, const u64 *__restrict__ dst_off,
                              const Intv *__restrict__ pool, ssq_smem_t *out)
{
	int r = blockIdx.x * blockDim.x + threadIdx.x;
	if (r >= n_reads) return;
	for (int i = 0; i < intv_cnt[r]; ++i) {
		const Intv p = pool[intv_off[r] + i];
		ssq_smem_t o; o.k = p.x0; o.l = p.x1; o.s = p.x2; o.qbeg = p.qb; o.qend = p.qe;
		out[dst_off[r] + i] = o;
	}
}

__global__ void k_gather_chains(int n_reads, const u64 *__restrict__ intv_off, const i32 *__restrict__ intv_cnt, const u64 *__restrict__ seed_off,
                                const ChainRec *__restrict__ outc, const Seed *__restrict__ sorted, const i32 *__restrict__ n_kept,
                                const u64 *__restrict__ chain_dst, const u64 *__restrict__ seed_dst, ssq_seed_t *seeds_out, u64 *chain_seed_off)
{
	int r = blockIdx.x * blockDim.x + threadIdx.x;
	if (r >= n_reads || n_kept[r] == 0) return;
	const u64 s0 = seed_off[intv_off[r]];
	u64 so = seed_dst[r];
	for (int c = 0; c < n_kept[r]; ++c) {
		const ChainRec ch = outc[s0 + c];
		chain_seed_off[chain_dst[r] + c] = so;
		for (int s = 0; s < ch.n; ++s) {
			const Seed x = sorted[s0 + ch.seed_start + s];
			ssq_seed_t o; o.rbeg = x.rbeg; o.qbeg = x.qbeg; o.len = x.len;
			seeds_out[so++] = o;
		}
	}
}

__global__ void k_widen_i32(int n, const i32 *in, u64 *out) { int i = blockIdx.x * blockDim.x + threadIdx.x; if (i < n) out[i] = (u64)in[i]; }
__global__ void k_widen_u32(u64 n, const u32 *in, u64 *out) { u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; if (i < n) out[i] = (u64)in[i]; }

// --------------------------------------------------------------------------- dup-mark ----
__global__ void k_dup_keys(u64 n, const ssq_dupsig_t *__restrict__ sig, u64 *key1, u64 *key2, u32 *idx)
{
	u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const ssq_dupsig_t s = sig[i];
	key1[i] = s.valid ? (s.pos1 << 1 | (s.strand1 & 1)) : ~0ull;
	key2[i] = s.valid ? (s.pos2 << 1 | (s.strand2 & 1)) : ~0ull;
	idx[i] = (u32)i;
}
__global__ void k_dup_gather(u64 n, const u32 *__restrict__ idx, const u64 *__restrict__ key1, u64 *key1g)
{
	u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
	if (i < n) key1g[i] = key1[idx[i]];
}
// after the two stable passes elements are ordered by (key1, key2, input ordinal): every element equal to its
// predecessor is a later occurrence of the same signature
__global__ void k_dup_mark(u64 n, const u32 *__restrict__ idx, const u64 *__restrict__ key1s, const u64 *__restrict__ key2, const ssq_dupsig_t *__restrict__ sig, uint8_t *is_dup)
{
	u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const u32 me = idx[i];
	uint8_t d = 0;
	if (i > 0 && sig[me].valid) {
		const u32 pv = idx[i - 1];
		d = sig[pv].valid && key1s[i] == key1s[i - 1] && key2[me] == key2[pv];
	}
	is_dup[me] = d;
}

// ===================================================================== host-side launch code ====
#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { ssq_set_error("%s:%d: %s", __FILE__, __LINE__, cudaGetErrorString(e_)); return SSQ_ECUDA; } } while (0)


struct ssq_batch {
	const ssq_index *idx;
	ssq_opts_t opt;
	int n_reads, max_len, n_sm;
	cudaStream_t st;
	DBuf seq, read_off, pool, scratch, intv_off, intv_cnt, l_rep, misc, nocc, seed_off, seeds;
	DBuf chain_of, ch, ord, wi, sorted, outc, n_kept, n_kseeds, task_off, tasks, cand, srt, regs, n_regs, reg_off, cubtmp, out;
	DBuf xinfo, xres[2], xwide, xkey[2], xidx[2], xretry, xmisc, xneed, xhave, xkp, xheavy, xsel, xlist[2], srt2, xgiant, xgiant2, xovf, scratch2, xowner, xp3, xp3n, xsplit, xstage, xmems, xmemr, xcalls, xfl, xk64[2], xi32[2];
	int ext_rounds; float select_ms;
	u64 n_intv, n_seeds, n_tasks, n_regs_total;
	u64 pool_cap;
	Counters h_cnt;
	int launches, own_stream, smem_variant;
	u64 call_cap = 0, fl_cap = 0; // split seeding: capacities of the call and forward-list pools
	cudaEvent_t ev[6], evc[4], evs[2], evx[2], evb[4]; /* evb: around the two backward-sweep launches of the split seeding */ // stage boundaries; chaining tiers; k_smem_m alone; selection kernels of one round // stage boundaries; chaining tiers (light start, heavy start, end)
	float stage_ms[5];
	ssq_batch() { memset(&h_cnt, 0, sizeof h_cnt); n_intv = n_seeds = n_tasks = n_regs_total = 0; launches = 0; own_stream = 1; pool_cap = 0; ext_rounds = 0; select_ms = 0.f; { const char *v = getenv("SSQ_SMEM_VARIANT"); smem_variant = v ? atoi(v) : 3; /* phase-split seeding (r02: 48.9 ms vs 59.9 ms for the state machine on the bench workload); indexes without bwt32 use the 64-bit state machine */ } memset(stage_ms, 0, sizeof stage_ms); }
};

// misc buffer layout (device): [0] pool_n (u64)  [1] work (int) + err (int)  [2..] Counters
struct Misc { unsigned long long pool_n; int work, err; unsigned int n_ovf, pad; Counters cnt; };

static int scan_u64(ssq_batch *b, const u64 *in, u64 *out, size_t n) // exclusive sum, out has n+1 entries (out[n] = total)
{
	size_t tmp = 0;
	cub::DeviceScan::ExclusiveSum(0, tmp, in, out, (int)n, b->st);
	if (b->cubtmp.need(tmp)) return SSQ_ENOMEM;
	CK(cub::DeviceScan::ExclusiveSum(b->cubtmp.p, tmp, in, out, (int)n, b->st));
	return 0;
}

extern "C" int ssq_batch_upload(ssq_batch_t *b, int n_reads, const uint8_t *seq, const uint64_t *read_off)
{
	if (!b || n_reads < 0 || !read_off || (n_reads > 0 && !seq)) return SSQ_EINVAL;
	int rc = ssq_use_device(b->idx->device);
	if (rc) return rc;
	b->n_reads = n_reads;
	b->max_len = 0;
	for (int i = 0; i < n_reads; ++i) { int l = (int)(read_off[i + 1] - read_off[i]); if (l > b->max_len) b->max_len = l; }
	if (b->max_len > SSQ_MAX_READ_LEN) { ssq_set_error("read longer than %d bases", SSQ_MAX_READ_LEN); return SSQ_ELEN; }
	const u64 total = read_off[n_reads];
	if (b->seq.need(total + 16) || b->read_off.need((size_t)(n_reads + 1) * 8)) return SSQ_ENOMEM;
	if (total) CK(cudaMemcpyAsync(b->seq.p, seq, total, cudaMemcpyHostToDevice, b->st));
	CK(cudaMemcpyAsync(b->read_off.p, read_off, (size_t)(n_reads + 1) * 8, cudaMemcpyHostToDevice, b->st));
	CK(cudaStreamSynchronize(b->st));
	b->n_intv = b->n_seeds = b->n_tasks = b->n_regs_total = 0;
	return SSQ_OK;
}

int ssq_batch_reserve(ssq_batch_t *b, int n_reads, u64 total_bases, int max_len, uint8_t **d_seq, u64 **d_off)
{
	if (!b || n_reads < 0) return SSQ_EINVAL;
	if (max_len > SSQ_MAX_READ_LEN) { ssq_set_error("read longer than %d bases", SSQ_MAX_READ_LEN); return SSQ_ELEN; }
	b->n_reads = n_reads; b->max_len = max_len;
	if (b->seq.need(total_bases + 16) || b->read_off.need((size_t)(n_reads + 1) * 8)) return SSQ_ENOMEM;
	b->n_intv = b->n_seeds = b->n_tasks = b->n_regs_total = 0;
	*d_seq = b->seq.as<uint8_t>(); *d_off = b->read_off.as<u64>();
	return SSQ_OK;
}

extern "C" int ssq_batch_create(const ssq_index_t *idx, const ssq_opts_t *opt, int n_reads, const uint8_t *seq, const uint64_t *read_off, ssq_batch_t **out)
{
	if (!idx || !opt || n_reads < 0 || !out) return SSQ_EINVAL;
	int rc = ssq_use_device(idx->device);
	if (rc) return rc;
	ssq_batch *b = new ssq_batch();
	b->idx = idx; b->opt = *opt; b->n_reads = 0; b->max_len = 0;
	cudaDeviceProp prop;
	CK(cudaGetDeviceProperties(&prop, idx->device));
	b->n_sm = prop.multiProcessorCount;
	CK(cudaStreamCreateWithFlags(&b->st, cudaStreamNonBlocking));
	for (int i = 0; i < 6; ++i) CK(cudaEventCreate(&b->ev[i]));
	for (int i = 0; i < 4; ++i) CK(cudaEventCreate(&b->evc[i]));
	for (int i = 0; i < 2; ++i) { CK(cudaEventCreate(&b->evs[i])); CK(cudaEventCreate(&b->evx[i])); }
	for (int i = 0; i < 4; ++i) CK(cudaEventCreate(&b->evb[i]));
	if (read_off && (rc = ssq_batch_upload(b, n_reads, seq, read_off))) { ssq_batch_free(b); return rc; }
	*out = b;
	return SSQ_OK;
}

extern "C" void ssq_batch_free(ssq_batch_t *b)
{
	if (!b) return;
	DBuf *all[] = {&b->seq, &b->read_off, &b->pool, &b->scratch, &b->intv_off, &b->intv_cnt, &b->l_rep, &b->misc, &b->nocc, &b->seed_off, &b->seeds,
	               &b->chain_of, &b->ch, &b->ord, &b->wi, &b->sorted, &b->outc, &b->n_kept, &b->n_kseeds, &b->task_off, &b->tasks, &b->cand, &b->srt,
	               &b->regs, &b->n_regs, &b->reg_off, &b->cubtmp, &b->out,
	               &b->xinfo, &b->xres[0], &b->xres[1], &b->xwide, &b->xkey[0], &b->xkey[1], &b->xidx[0], &b->xidx[1], &b->xretry, &b->xmisc, &b->xneed, &b->xhave, &b->xkp, &b->xheavy, &b->xsel, &b->xlist[0], &b->xlist[1], &b->srt2, &b->xgiant, &b->xgiant2, &b->xovf, &b->scratch2, &b->xowner, &b->xp3, &b->xp3n, &b->xsplit, &b->xstage, &b->xmems, &b->xmemr, &b->xcalls, &b->xfl, &b->xk64[0], &b->xk64[1], &b->xi32[0], &b->xi32[1]};
	for (size_t i = 0; i < sizeof(all) / sizeof(all[0]); ++i) all[i]->release();
	for (int i = 0; i < 6; ++i) cudaEventDestroy(b->ev[i]);
	for (int i = 0; i < 4; ++i) cudaEventDestroy(b->evc[i]);
	for (int i = 0; i < 2; ++i) { cudaEventDestroy(b->evs[i]); cudaEventDestroy(b->evx[i]); }
	for (int i = 0; i < 4; ++i) cudaEventDestroy(b->evb[i]);
	if (b->own_stream) cudaStreamDestroy(b->st);
	delete b;
}

BatchView ssq_batch_view(ssq_batch_t *b)
{
	BatchView v;
	v.ix = b->idx->dev; v.n_reads = b->n_reads; v.n_sm = b->n_sm;
	v.seq = b->seq.as<uint8_t>(); v.read_off = b->read_off.as<u64>();
	v.task_off = b->task_off.as<u64>(); v.n_regs = b->n_regs.as<u32>(); v.regs = b->regs.as<RegCand>();
	return v;
}
extern "C" void *ssq_batch_stream(ssq_batch_t *b) { return (void*)b->st; }
extern "C" int ssq_batch_set_stream(ssq_batch_t *b, void *stream)
{
	if (!b || !stream) return SSQ_EINVAL;
	if (b->own_stream) cudaStreamDestroy(b->st);
	b->st = (cudaStream_t)stream; b->own_stream = 0;
	return SSQ_OK;
}
extern "C" int ssq_batch_sync(ssq_batch_t *b) { CK(cudaStreamSynchronize(b->st)); return SSQ_OK; }

// stage A, phase-split form (SSQ_SMEM_VARIANT=3; indexes with bwt32): see the kernels' header comment
static int run_smem_split(ssq_batch *b)
{
	const int n = b->n_reads, lcap = b->max_len > 0 ? b->max_len : 1;
	const char *lc_env = getenv("SSQ_LIST_CAP");
	const int list_cap = lc_env ? atoi(lc_env) : 6;
	const int fgrid = b->n_sm * 5, bgrid = b->n_sm * 8, bthreads = 128; // persistent lanes; the grid may exceed what is resident
	const int scratch_cap = lcap + 1; // a call cannot keep more intervals than the read has positions
	if (b->intv_off.need((size_t)(n + 1) * 8) || b->intv_cnt.need((size_t)(n + 1) * 4) || b->l_rep.need((size_t)(n + 1) * 4) || b->misc.need(sizeof(Misc)) ||
	    b->xsplit.need(sizeof(Split))) return SSQ_ENOMEM;
	if (b->xstage.need((size_t)fgrid * 256 * (size_t)(lcap + 1) * sizeof(FwdEntry))) return SSQ_ENOMEM;
	if (b->scratch.need((size_t)bgrid * bthreads * ((size_t)scratch_cap + (size_t)(lcap + 1)) * sizeof(Intv))) return SSQ_ENOMEM;
	const int p3_stride = lcap / (b->opt.min_seed_len + 1) + 2;
	const bool with_p3 = b->opt.max_mem_intv > 0;
	if (with_p3 && (b->xp3.need((size_t)n * p3_stride * sizeof(Intv)) || b->xp3n.need((size_t)(n + 1) * 4))) return SSQ_ENOMEM;
	if (getenv("SSQ_SPLIT_TINY_POOLS") && b->call_cap == 0) { b->pool_cap = 256; b->call_cap = 64; b->fl_cap = 512; } // tests: force the overflow retry
	if (b->pool_cap == 0) b->pool_cap = (u64)n * 48 + 4096;
	if (b->call_cap == 0) b->call_cap = (u64)n * 10 + 4096;
	if (b->fl_cap == 0) b->fl_cap = (u64)n * 96 + 65536;
	const bool lean = b->smem_variant == 4;
	const int lean_blocks = getenv("SSQ_SMEM_BLOCKS") ? atoi(getenv("SSQ_SMEM_BLOCKS")) : 8;
	typedef void (*bwd_kernel_t)(DevIndex, ssq_opts_t, const uint8_t*, const u64*, int, int, Intv*, int, const SeedCall*, const FwdEntry*, int, Intv*, u32*, u64, Split*, Counters*);
	const int bwd_blocks = getenv("SSQ_SMEM_BWD_BLOCKS") ? atoi(getenv("SSQ_SMEM_BWD_BLOCKS")) : 6; // resident blocks per SM the backward kernel is compiled for (register budget)
	const bwd_kernel_t kb = bwd_blocks >= 8 ? k_smem_bwd<8> : bwd_blocks == 7 ? k_smem_bwd<7> : k_smem_bwd<6>;
	CK(cudaFuncSetAttribute(kb, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)((size_t)bthreads * 2 * (list_cap > 0 ? list_cap : 1) * sizeof(uint4))));
	const bool tab = b->idx->dev.kmer_k > 0; // k-mer jump-start table loaded (SSQ_KMER_K): forward walks, the greedy pass and the lean backward kernel use it
	typedef void (*fwd_kernel_t)(DevIndex, ssq_opts_t, int, const uint8_t*, const u64*, int, FwdEntry*, SeedCall*, u64, FwdEntry*, u64, Split*, Counters*);
	typedef void (*bwd2_kernel_t)(DevIndex, ssq_opts_t, const uint8_t*, int, int, Intv*, int, const SeedCall*, const FwdEntry*, int, Intv*, u32*, u64, Split*, Counters*);
	const fwd_kernel_t kf1 = tab ? k_smem_fwd<1, true> : k_smem_fwd<1, false>, kf2 = tab ? k_smem_fwd<2, true> : k_smem_fwd<2, false>;
	const bwd2_kernel_t kb2 = lean_blocks >= 8 ? (tab ? k_smem_bwd2<8, true> : k_smem_bwd2<8, false>) : (tab ? k_smem_bwd2<6, true> : k_smem_bwd2<6, false>);
	CK(cudaFuncSetAttribute(kb2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)((size_t)bthreads * 2 * (list_cap > 0 ? list_cap : 1) * sizeof(uint4))));
	const size_t lsm = (size_t)bthreads * 2 * list_cap * sizeof(uint4);
	Misc *dm = b->misc.as<Misc>();
	Split *sp = b->xsplit.as<Split>();
	for (int attempt = 0; attempt < 12; ++attempt) {
		if (b->xmems.need(b->pool_cap * sizeof(Intv)) || b->xmemr.need(b->pool_cap * 4) || b->xcalls.need(b->call_cap * sizeof(SeedCall)) || b->xfl.need(b->fl_cap * sizeof(FwdEntry))) return SSQ_ENOMEM;
		CK(cudaMemsetAsync(b->misc.p, 0, sizeof(Misc), b->st));
		CK(cudaMemsetAsync(b->xsplit.p, 0, sizeof(Split), b->st));
		if (with_p3 && tab) k_smem_p3<u32, true><<<b->n_sm * 8, 256, 0, b->st>>>(b->idx->dev, b->opt, n, b->seq.as<uint8_t>(), b->read_off.as<u64>(), p3_stride, b->xp3.as<Intv>(), b->xp3n.as<i32>(), &dm->work, &dm->cnt);
		else if (with_p3) k_smem_p3<u32, false><<<b->n_sm * 8, 256, 0, b->st>>>(b->idx->dev, b->opt, n, b->seq.as<uint8_t>(), b->read_off.as<u64>(), p3_stride, b->xp3.as<Intv>(), b->xp3n.as<i32>(), &dm->work, &dm->cnt);
		kf1<<<fgrid, 256, 0, b->st>>>(b->idx->dev, b->opt, n, b->seq.as<uint8_t>(), b->read_off.as<u64>(), lcap, b->xstage.as<FwdEntry>(), b->xcalls.as<SeedCall>(), b->call_cap,
		                                       b->xfl.as<FwdEntry>(), b->fl_cap, sp, &dm->cnt);
		k_smem_snapshot<<<1, 1, 0, b->st>>>(sp, b->call_cap, b->pool_cap, 1); // n_calls1 = pass-1 calls (n_mems1 still 0)
		k_cnt_mark<<<1, 1, 0, b->st>>>(&dm->cnt, 8); CK(cudaEventRecord(b->evb[0], b->st));
		if (!lean) kb<<<bgrid, bthreads, lsm, b->st>>>(b->idx->dev, b->opt, b->seq.as<uint8_t>(), b->read_off.as<u64>(), lcap, list_cap, b->scratch.as<Intv>(), scratch_cap,
		                                             b->xcalls.as<SeedCall>(), b->xfl.as<FwdEntry>(), 0, b->xmems.as<Intv>(), b->xmemr.as<u32>(), b->pool_cap, sp, &dm->cnt);
		else kb2<<<bgrid, bthreads, lsm, b->st>>>(b->idx->dev, b->opt, b->seq.as<uint8_t>(), lcap, list_cap, b->scratch.as<Intv>(), scratch_cap,
		                                             b->xcalls.as<SeedCall>(), b->xfl.as<FwdEntry>(), 0, b->xmems.as<Intv>(), b->xmemr.as<u32>(), b->pool_cap, sp, &dm->cnt);
		CK(cudaEventRecord(b->evb[1], b->st)); k_cnt_mark<<<1, 1, 0, b->st>>>(&dm->cnt, 9);
		k_smem_snapshot<<<1, 1, 0, b->st>>>(sp, b->call_cap, b->pool_cap, 1); // n_mems1 = pass-1 intervals; n_calls1 unchanged (no calls were added)
		k_smem_p2sel<<<b->n_sm * 8, 256, 0, b->st>>>(b->opt, b->seq.as<uint8_t>(), b->read_off.as<u64>(), b->xmems.as<Intv>(), b->xmemr.as<u32>(), b->xcalls.as<SeedCall>(), b->call_cap, sp);
		k_smem_snapshot<<<1, 1, 0, b->st>>>(sp, b->call_cap, b->pool_cap, 0); // clamp the request range
		kf2<<<fgrid, 256, 0, b->st>>>(b->idx->dev, b->opt, n, b->seq.as<uint8_t>(), b->read_off.as<u64>(), lcap, b->xstage.as<FwdEntry>(), b->xcalls.as<SeedCall>(), b->call_cap,
		                                       b->xfl.as<FwdEntry>(), b->fl_cap, sp, &dm->cnt);
		k_cnt_mark<<<1, 1, 0, b->st>>>(&dm->cnt, 10); CK(cudaEventRecord(b->evb[2], b->st));
		if (!lean) kb<<<bgrid, bthreads, lsm, b->st>>>(b->idx->dev, b->opt, b->seq.as<uint8_t>(), b->read_off.as<u64>(), lcap, list_cap, b->scratch.as<Intv>(), scratch_cap,
		                                             b->xcalls.as<SeedCall>(), b->xfl.as<FwdEntry>(), 1, b->xmems.as<Intv>(), b->xmemr.as<u32>(), b->pool_cap, sp, &dm->cnt);
		else kb2<<<bgrid, bthreads, lsm, b->st>>>(b->idx->dev, b->opt, b->seq.as<uint8_t>(), lcap, list_cap, b->scratch.as<Intv>(), scratch_cap,
		                                             b->xcalls.as<SeedCall>(), b->xfl.as<FwdEntry>(), 1, b->xmems.as<Intv>(), b->xmemr.as<u32>(), b->pool_cap, sp, &dm->cnt);
		CK(cudaEventRecord(b->evb[3], b->st)); k_cnt_mark<<<1, 1, 0, b->st>>>(&dm->cnt, 11);
		if (with_p3) k_smem_p3_append<<<(n + 255) / 256, 256, 0, b->st>>>(n, b->xp3.as<Intv>(), b->xp3n.as<i32>(), p3_stride, b->xmems.as<Intv>(), b->xmemr.as<u32>(), b->pool_cap, sp);
		b->launches += 10;
		CK(cudaGetLastError());
		Split hs;
		CK(cudaMemcpyAsync(&hs, sp, sizeof(Split), cudaMemcpyDeviceToHost, b->st));
		CK(cudaStreamSynchronize(b->st));
		if (hs.err == 2) { // a pool was too small; the counters are lower bounds of what is needed
			if (hs.n_mems + 1 > b->pool_cap) b->pool_cap = hs.n_mems + hs.n_mems / 2 + 4096; else b->pool_cap += b->pool_cap / 2;
			{ const u64 nc = hs.need_calls > hs.n_calls ? hs.need_calls : hs.n_calls; if (nc + 1 > b->call_cap) b->call_cap = nc + nc / 2 + 4096; else b->call_cap += b->call_cap / 2; }
			if (hs.n_fl + 1 > b->fl_cap) b->fl_cap = hs.n_fl + hs.n_fl / 2 + 65536; else b->fl_cap += b->fl_cap / 2;
			continue;
		}
		if (hs.err) { ssq_set_error(hs.err == 3 ? "read longer than the kernel's length cap" : "seeding (split): a call overflowed its scratch"); return hs.err == 3 ? SSQ_ELEN : SSQ_ECAP; }
		const u64 N = hs.n_mems;
		b->n_intv = N;
		CK(cudaMemsetAsync(b->intv_off.p, 0, (size_t)(n + 1) * 8, b->st));
		CK(cudaMemsetAsync(b->intv_cnt.p, 0, (size_t)(n + 1) * 4, b->st));
		if (b->pool.need((N + 1) * sizeof(Intv))) return SSQ_ENOMEM;
		if (N) {
			if (N >= 0xffffffffull) { ssq_set_error("more than 2^32 seed intervals in one batch"); return SSQ_ECAP; }
			if (b->xk64[0].need(N * 8) || b->xk64[1].need(N * 8) || b->xi32[0].need(N * 4) || b->xi32[1].need(N * 4)) return SSQ_ENOMEM;
			k_smem_keys<<<(unsigned)((N + 255) / 256), 256, 0, b->st>>>(N, b->xmems.as<Intv>(), b->xmemr.as<u32>(), b->xk64[0].as<u64>(), b->xi32[0].as<u32>());
			int rbits = 1; while ((1ull << rbits) < (u64)n + 1) ++rbits;
			size_t tb = 0;
			cub::DeviceRadixSort::SortPairs(0, tb, b->xk64[0].as<u64>(), b->xk64[1].as<u64>(), b->xi32[0].as<u32>(), b->xi32[1].as<u32>(), (int)N, 0, 16 + rbits, b->st);
			if (b->cubtmp.need(tb)) return SSQ_ENOMEM;
			CK(cub::DeviceRadixSort::SortPairs(b->cubtmp.p, tb, b->xk64[0].as<u64>(), b->xk64[1].as<u64>(), b->xi32[0].as<u32>(), b->xi32[1].as<u32>(), (int)N, 0, 16 + rbits, b->st));
			k_smem_publish<<<(unsigned)((N + 255) / 256), 256, 0, b->st>>>(N, b->xk64[1].as<u64>(), b->xi32[1].as<u32>(), b->xmems.as<Intv>(), b->pool.as<Intv>(), b->intv_off.as<u64>(), b->intv_cnt.as<i32>());
			b->launches += 3;
		}
		k_smem_lrep<<<(n + 255) / 256, 256, 0, b->st>>>(n, b->opt, b->pool.as<Intv>(), b->intv_off.as<u64>(), b->intv_cnt.as<i32>(), b->l_rep.as<i32>());
		++b->launches;
		CK(cudaGetLastError());
		return SSQ_OK;
	}
	ssq_set_error("seeding (split): pools kept overflowing");
	return SSQ_ECAP;
}

// stage A: seeding (+ pool overflow retry). leaves intervals in pool, per-read (intv_off, intv_cnt, l_rep)
static int run_smem(ssq_batch *b)
{
	const int n = b->n_reads, lcap = b->max_len > 0 ? b->max_len : 1;
	if ((b->smem_variant == 3 || b->smem_variant == 4) && b->idx->dev.bwt32 && n > 0) return run_smem_split(b);
	const int variant = b->smem_variant >= 3 ? 2 : b->smem_variant;
	const int warps_per_block = 4, threads = warps_per_block * 32;
	const size_t smem = variant == 0 ? (size_t)warps_per_block * 2 * (lcap + 1) * sizeof(Intv) : 0;
	const char *lc_env = getenv("SSQ_LIST_CAP");
	// shared-memory list entries per lane.  Measured (profiles/r01_smem_sweep.txt): the 32-bit machine is fastest with 6 blocks/SM and
	// short lists — what the lists do not take stays L1 for the query bytes, the output list and the overflow entries
	const bool m32_ = variant == 2 && b->idx->dev.bwt32 != 0 && !getenv("SSQ_SMEM_M64");
	const int list_cap = variant == 2 && b->idx->dev.seq_len < 0xffffffffull ? (lc_env ? atoi(lc_env) : m32_ ? 6 : 10) : 0;
	// 32-bit machine (indexes with bwt32): fewer registers, so more blocks per SM when the shared-memory lists leave room for them
	const bool m32 = m32_;
	const int minb = m32 ? (getenv("SSQ_SMEM_BLOCKS") ? atoi(getenv("SSQ_SMEM_BLOCKS")) : 6) : 5;
	typedef void (*smem_kernel_t)(DevIndex, ssq_opts_t, int, const uint8_t*, const u64*, int, int, int, Intv*, int, Intv*, u64, unsigned long long*, u64*, i32*, i32*, int*, int*, Counters*, const u32*, u32*, unsigned int*, const Intv*, const i32*, int);
	const bool mtab = m32 && b->idx->dev.kmer_k > 0; // SSQ_KMER_K loaded the k-mer jump-start table
	const smem_kernel_t km = !m32 ? k_smem_m<u64, 5, false> : mtab ? k_smem_m<u32, 6, true> : minb >= 8 ? k_smem_m<u32, 8, false> : minb == 7 ? k_smem_m<u32, 7, false> : minb == 6 ? k_smem_m<u32, 6, false> : k_smem_m<u32, 5, false>;
	if (variant == 2) CK(cudaFuncSetAttribute(km, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)((size_t)threads * 2 * (list_cap > 0 ? list_cap : 1) * sizeof(uint4))));
	int blocks_per_sm = variant == 0 ? (int)((200 * 1024) / (smem + 1024)) : 8;
	if (blocks_per_sm > 8) blocks_per_sm = 8;
	if (blocks_per_sm < 1) blocks_per_sm = 1;
	const int grid = b->n_sm * blocks_per_sm;
	const int scratch_cap = variant == 0 ? 2048 : 768;
	const size_t scratch_entries = variant == 0 ? (size_t)grid * warps_per_block * scratch_cap : (size_t)grid * threads * ((size_t)scratch_cap + 2 * (size_t)(lcap + 1) + (size_t)(scratch_cap + 7) / 8);
	if (b->pool_cap == 0) b->pool_cap = (u64)n * 48 + 4096;
	if (b->scratch.need(scratch_entries * sizeof(Intv))) return SSQ_ENOMEM;
	if (b->intv_off.need((size_t)(n + 1) * 8) || b->intv_cnt.need((size_t)(n + 1) * 4) || b->l_rep.need((size_t)(n + 1) * 4) || b->misc.need(sizeof(Misc)) || b->xovf.need((size_t)(n + 1) * 4)) return SSQ_ENOMEM;
	if (variant == 0) CK(cudaFuncSetAttribute(k_smem, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
	for (int attempt = 0; attempt < 6; ++attempt) {
		if (b->pool.need(b->pool_cap * sizeof(Intv))) return SSQ_ENOMEM;
		CK(cudaMemsetAsync(b->misc.p, 0, sizeof(Misc), b->st));
		Misc *dm = b->misc.as<Misc>();
		const Intv *p3buf = 0; const i32 *p3cnt = 0;
		const int p3_stride = lcap / (b->opt.min_seed_len + 1) + 2;
		if (variant == 2 && b->opt.max_mem_intv > 0) {
			if (b->xp3.need((size_t)n * p3_stride * sizeof(Intv)) || b->xp3n.need((size_t)(n + 1) * 4)) return SSQ_ENOMEM;
			if (mtab) k_smem_p3<u32, true><<<b->n_sm * 8, 256, 0, b->st>>>(b->idx->dev, b->opt, n, b->seq.as<uint8_t>(), b->read_off.as<u64>(), p3_stride, b->xp3.as<Intv>(), b->xp3n.as<i32>(), &dm->work, &dm->cnt);
			else if (m32) k_smem_p3<u32, false><<<b->n_sm * 8, 256, 0, b->st>>>(b->idx->dev, b->opt, n, b->seq.as<uint8_t>(), b->read_off.as<u64>(), p3_stride, b->xp3.as<Intv>(), b->xp3n.as<i32>(), &dm->work, &dm->cnt);
			else k_smem_p3<u64, false><<<b->n_sm * 8, 256, 0, b->st>>>(b->idx->dev, b->opt, n, b->seq.as<uint8_t>(), b->read_off.as<u64>(), p3_stride, b->xp3.as<Intv>(), b->xp3n.as<i32>(), &dm->work, &dm->cnt);
			CK(cudaMemsetAsync(&dm->work, 0, 4, b->st));
			++b->launches;
			p3buf = b->xp3.as<Intv>(); p3cnt = b->xp3n.as<i32>();
		}
		if (variant == 0)
			k_smem<<<grid, threads, smem, b->st>>>(b->idx->dev, b->opt, n, b->seq.as<uint8_t>(), b->read_off.as<u64>(), lcap, b->scratch.as<Intv>(), scratch_cap,
			                                      b->pool.as<Intv>(), b->pool_cap, &dm->pool_n, b->intv_off.as<u64>(), b->intv_cnt.as<i32>(), b->l_rep.as<i32>(), &dm->work, &dm->err, &dm->cnt);
		else if (variant == 2) {
			CK(cudaEventRecord(b->evs[0], b->st));
			km<<<grid, threads, (size_t)threads * 2 * list_cap * sizeof(uint4), b->st>>>(b->idx->dev, b->opt, n, b->seq.as<uint8_t>(), b->read_off.as<u64>(), lcap, list_cap, getenv("SSQ_SLOW_BATCH") ? atoi(getenv("SSQ_SLOW_BATCH")) : 8, b->scratch.as<Intv>(), scratch_cap,
			                                     b->pool.as<Intv>(), b->pool_cap, &dm->pool_n, b->intv_off.as<u64>(), b->intv_cnt.as<i32>(), b->l_rep.as<i32>(), &dm->work, &dm->err, &dm->cnt,
			                                     (const u32*)0, b->xovf.as<u32>(), &dm->n_ovf, p3buf, p3cnt, p3_stride);
			CK(cudaEventRecord(b->evs[1], b->st));
		} else
			k_smem_t<<<grid, threads, 0, b->st>>>(b->idx->dev, b->opt, n, b->seq.as<uint8_t>(), b->read_off.as<u64>(), lcap, b->scratch.as<Intv>(), scratch_cap,
			                                     b->pool.as<Intv>(), b->pool_cap, &dm->pool_n, b->intv_off.as<u64>(), b->intv_cnt.as<i32>(), b->l_rep.as<i32>(), &dm->work, &dm->err, &dm->cnt);
		++b->launches;
		CK(cudaGetLastError());
		Misc hm;
		CK(cudaMemcpyAsync(&hm, b->misc.p, sizeof(Misc), cudaMemcpyDeviceToHost, b->st));
		CK(cudaStreamSynchronize(b->st));
		if (variant == 2 && hm.err == 0 && hm.n_ovf) { // low-complexity reads with more intervals than a lane's scratch holds: again, few lanes, big scratch
			const int cap2 = 16384, grid2 = 8;
			const size_t per2 = (size_t)cap2 + 2 * (size_t)(lcap + 1) + (size_t)(cap2 + 7) / 8;
			if (b->scratch2.need((size_t)grid2 * threads * per2 * sizeof(Intv))) return SSQ_ENOMEM;
			CK(cudaMemsetAsync(&dm->work, 0, 4, b->st));
			km<<<grid2, threads, (size_t)threads * 2 * list_cap * sizeof(uint4), b->st>>>(b->idx->dev, b->opt, (int)hm.n_ovf, b->seq.as<uint8_t>(), b->read_off.as<u64>(), lcap, list_cap, 1, b->scratch2.as<Intv>(), cap2,
			        b->pool.as<Intv>(), b->pool_cap, &dm->pool_n, b->intv_off.as<u64>(), b->intv_cnt.as<i32>(), b->l_rep.as<i32>(), &dm->work, &dm->err, &dm->cnt,
			        b->xovf.as<u32>(), (u32*)0, (unsigned int*)0, p3buf, p3cnt, p3_stride);
			++b->launches;
			CK(cudaGetLastError());
			CK(cudaMemcpyAsync(&hm, b->misc.p, sizeof(Misc), cudaMemcpyDeviceToHost, b->st));
			CK(cudaStreamSynchronize(b->st));
		}
		if (hm.err == 0) { b->n_intv = hm.pool_n; return SSQ_OK; }
		if (hm.err == 2) { b->pool_cap = hm.pool_n + hm.pool_n / 8 + 4096; continue; } // pool too small: its true size is now known
		ssq_set_error(hm.err == 3 ? "read longer than the kernel's length cap" : "a read produced more than %d seed intervals", scratch_cap);
		return hm.err == 3 ? SSQ_ELEN : SSQ_ECAP;
	}
	ssq_set_error("interval pool kept overflowing");
	return SSQ_ECAP;
}

// stage B: SA look-ups -> seeds (read-contiguous)
static int run_sa(ssq_batch *b)
{
	const u64 ni = b->n_intv;
	if (b->nocc.need((ni + 1) * 4) || b->seed_off.need((ni + 2) * 8) || b->tasks.need((ni + 1) * 8)) return SSQ_ENOMEM; // tasks reused as temp u64
	b->n_seeds = 0;
	if (ni == 0) { CK(cudaMemsetAsync(b->seed_off.p, 0, 16, b->st)); return SSQ_OK; }
	k_occ_count<<<(unsigned)((ni + 255) / 256), 256, 0, b->st>>>(b->pool.as<Intv>(), ni, b->opt.max_occ, b->nocc.as<u32>());
	k_widen_u32<<<(unsigned)((ni + 255) / 256), 256, 0, b->st>>>(ni, b->nocc.as<u32>(), b->tasks.as<u64>());
	b->launches += 2;
	int rc = scan_u64(b, b->tasks.as<u64>(), b->seed_off.as<u64>(), ni + 1); // ni+1 inputs so that out[ni] = total (input[ni] is ignored garbage)
	if (rc) return rc;
	++b->launches;
	CK(cudaMemcpyAsync(&b->n_seeds, b->seed_off.as<u64>() + ni, 8, cudaMemcpyDeviceToHost, b->st));
	CK(cudaStreamSynchronize(b->st));
	if (b->seeds.need((b->n_seeds + 1) * sizeof(Seed))) return SSQ_ENOMEM;
	if (b->n_seeds) {
		if (ni >= 0xffffffffull) { ssq_set_error("more than 2^32 seed intervals in one batch"); return SSQ_ECAP; }
		if (b->xowner.need((b->n_seeds + 1) * 4)) return SSQ_ENOMEM;
		CK(cudaMemsetAsync(b->xowner.p, 0, b->n_seeds * 4, b->st));
		k_sa_owner<<<(unsigned)((ni + 255) / 256), 256, 0, b->st>>>(ni, b->seed_off.as<u64>(), b->xowner.as<u32>());
		size_t tb = 0;
		cub::DeviceScan::InclusiveScan(0, tb, b->xowner.as<u32>(), b->xowner.as<u32>(), cub::Max(), (int)b->n_seeds, b->st);
		if (b->cubtmp.need(tb)) return SSQ_ENOMEM;
		CK(cub::DeviceScan::InclusiveScan(b->cubtmp.p, tb, b->xowner.as<u32>(), b->xowner.as<u32>(), cub::Max(), (int)b->n_seeds, b->st));
		k_sa<<<(unsigned)((b->n_seeds + 255) / 256), 256, 0, b->st>>>(b->idx->dev, b->opt, b->pool.as<Intv>(), b->seed_off.as<u64>(), b->xowner.as<u32>(), b->n_seeds, b->seeds.as<Seed>(),
		                                                               &b->misc.as<Misc>()->cnt);
		b->launches += 3;
		CK(cudaGetLastError());
	}
	return SSQ_OK;
}

// The cut between the thread-per-read and the warp-per-read tier of a stage (work items per read), overridable for tests.
// Measured on B200 (profiles/r01_tier_sweep.txt): the stage time is flat between 32 and 64 and grows on either side.
static int tier_threshold(ssq_batch *b, const char *env, int dflt, int *d_thresh)
{
	const int v = getenv(env) ? atoi(getenv(env)) : dflt;
	CK(cudaMemcpyAsync(d_thresh, &v, 4, cudaMemcpyHostToDevice, b->st));
	CK(cudaStreamSynchronize(b->st)); // v is on the stack
	return SSQ_OK;
}

// stage C: chaining + filter
static int run_chain(ssq_batch *b)
{
	const int n = b->n_reads;
	const u64 ns = b->n_seeds + 1;
	if (b->chain_of.need(ns * 4) || b->ch.need(ns * sizeof(ChainRec)) || b->ord.need(ns * 4) || b->wi.need(ns * sizeof(WIdx)) || b->sorted.need(ns * sizeof(Seed)) ||
	    b->outc.need(ns * sizeof(ChainRec)) || b->xkp.need(ns * sizeof(KeptChain)) || b->n_kept.need((size_t)(n + 1) * 4) || b->n_kseeds.need((size_t)(n + 1) * 4)) return SSQ_ENOMEM;
	if (n) {
		if (b->xheavy.need((size_t)(n + 1) * 4) || b->xmisc.need(256)) return SSQ_ENOMEM;
		unsigned int *n_heavy = b->xmisc.as<unsigned int>() + 24;
		int *heavy_thresh = b->xmisc.as<int>() + 27;
		const int rc = tier_threshold(b, "SSQ_HEAVY_SEEDS", 16, heavy_thresh);
		if (rc) return rc;
		CK(cudaMemsetAsync(n_heavy, 0, 8, b->st));
		CK(cudaMemsetAsync(&b->misc.as<Misc>()->work, 0, 4, b->st));
		CK(cudaEventRecord(b->evc[0], b->st));
		k_chain<<<b->n_sm * 12, 128, 0, b->st>>>(b->idx->dev, b->opt, n, b->read_off.as<u64>(), b->intv_off.as<u64>(), b->intv_cnt.as<i32>(), b->l_rep.as<i32>(),
		                                           b->seed_off.as<u64>(), b->seeds.as<Seed>(), b->chain_of.as<i32>(), b->ch.as<ChainRec>(), b->ord.as<i32>(), b->wi.as<WIdx>(),
		                                           b->sorted.as<Seed>(), b->outc.as<ChainRec>(), b->xkp.as<KeptChain>(), b->n_kept.as<i32>(), b->n_kseeds.as<u32>(), &b->misc.as<Misc>()->work, &b->misc.as<Misc>()->cnt, heavy_thresh, b->xheavy.as<u32>(), n_heavy);
		CK(cudaMemsetAsync(&b->misc.as<Misc>()->work, 0, 4, b->st));
		CK(cudaEventRecord(b->evc[1], b->st));
		// warp-per-read tiers: a small shared-memory footprint first (many warps per SM); what overflows is retried with 4x the
		// capacity, and what overflows that with a whole SM's shared memory per warp
		{
			static const int caps[3] = {getenv("SSQ_COOP_CAP") ? atoi(getenv("SSQ_COOP_CAP")) : 256, 1024, 4608};
			unsigned int *n_lvl[3] = {n_heavy, n_heavy + 1, b->xmisc.as<unsigned int>() + 29};
			if (b->xgiant.need((size_t)(n + 1) * 4) || b->xgiant2.need((size_t)(n + 1) * 4)) return SSQ_ENOMEM;
			u32 *lists[3] = {b->xheavy.as<u32>(), b->xgiant.as<u32>(), b->xgiant2.as<u32>()};
			CK(cudaMemsetAsync(n_lvl[2], 0, 4, b->st));
			CK(cudaFuncSetAttribute(k_chain_coop, cudaFuncAttributeMaxDynamicSharedMemorySize, 48 * caps[2]));
			for (int lvl = 0; lvl < 3; ++lvl) {
				if (lvl == 1) CK(cudaEventRecord(b->evc[3], b->st));
				const int fit = (int)(220 * 1024 / (48 * caps[lvl] + 1024));
				const int per_sm = fit < 1 ? 1 : fit > 24 ? 24 : fit;
				CK(cudaMemsetAsync(&b->misc.as<Misc>()->work, 0, 4, b->st));
				k_chain_coop<<<b->n_sm * per_sm, 32, 48 * caps[lvl], b->st>>>(b->idx->dev, b->opt, caps[lvl], b->read_off.as<u64>(), b->intv_off.as<u64>(), b->intv_cnt.as<i32>(), b->l_rep.as<i32>(),
				        b->seed_off.as<u64>(), b->seeds.as<Seed>(), b->chain_of.as<i32>(), b->ch.as<ChainRec>(), b->ord.as<i32>(), b->wi.as<WIdx>(),
				        b->sorted.as<Seed>(), b->outc.as<ChainRec>(), b->xkp.as<KeptChain>(), b->n_kept.as<i32>(), b->n_kseeds.as<u32>(), &b->misc.as<Misc>()->work,
				        lists[lvl], n_lvl[lvl], lvl < 2 ? lists[lvl + 1] : (u32*)0, lvl < 2 ? n_lvl[lvl + 1] : (unsigned int*)0);
				++b->launches;
			}
		}
		CK(cudaEventRecord(b->evc[2], b->st));
		++b->launches;
		CK(cudaGetLastError());
	}
	return SSQ_OK;
}

// stage D: task list + extension ; stage E: selection
static int run_extend(ssq_batch *b)
{
	const int n = b->n_reads;
	if (b->task_off.need((size_t)(n + 2) * 8) || b->reg_off.need((size_t)(n + 2) * 8) || b->n_regs.need((size_t)(n + 1) * 4)) return SSQ_ENOMEM;
	b->n_tasks = 0;
	if (n == 0) return SSQ_OK;
	// reg_off used as a temp for the widened counts
	k_widen_u32<<<(n + 255) / 256, 256, 0, b->st>>>((u64)n, b->n_kseeds.as<u32>(), b->reg_off.as<u64>());
	int rc = scan_u64(b, b->reg_off.as<u64>(), b->task_off.as<u64>(), (size_t)n + 1);
	if (rc) return rc;
	b->launches += 2;
	CK(cudaMemcpyAsync(&b->n_tasks, b->task_off.as<u64>() + n, 8, cudaMemcpyDeviceToHost, b->st));
	CK(cudaStreamSynchronize(b->st));
	const u64 nt = b->n_tasks;
	if (b->tasks.need((nt + 1) * sizeof(Task)) || b->cand.need((nt + 1) * sizeof(RegCand)) || b->srt.need((nt + 1) * 8) || b->regs.need((nt + 1) * sizeof(RegCand))) return SSQ_ENOMEM;
	if (b->xinfo.need((nt + 1) * sizeof(ExtInfo)) || b->xres[0].need((nt + 1) * sizeof(ExtRes)) || b->xres[1].need((nt + 1) * sizeof(ExtRes)) || b->xwide.need(2 * (nt + 1)) ||
	    b->xkey[0].need((nt + 1) * 4) || b->xkey[1].need((nt + 1) * 4) || b->xidx[0].need((nt + 1) * 4) || b->xidx[1].need((nt + 1) * 4) || b->xretry.need((nt + 1) * 4) ||
	    b->xmisc.need(256)) return SSQ_ENOMEM;
	if (b->xneed.need(nt + 1) || b->xhave.need(nt + 1) || b->xsel.need((size_t)(n + 1) * sizeof(SelState)) || b->xlist[0].need((size_t)(n + 1) * 4) || b->xlist[1].need((size_t)(n + 1) * 4) ||
	    b->srt2.need((nt + 1) * 8) || b->xheavy.need((size_t)(n + 1) * 4)) return SSQ_ENOMEM;
	CK(cudaEventRecord(b->ev[3], b->st));
	float ms_sel = 0.f;
	if (nt) {
		k_tasks<<<(n + 255) / 256, 256, 0, b->st>>>(n, b->intv_off.as<u64>(), b->intv_cnt.as<i32>(), b->seed_off.as<u64>(), b->outc.as<ChainRec>(), b->n_kept.as<i32>(),
		                                           b->task_off.as<u64>(), b->tasks.as<Task>());
		const unsigned G = (unsigned)((nt + 255) / 256);
		uint8_t *wide_l = b->xwide.as<uint8_t>(), *wide_r = wide_l + (nt + 1), *need = b->xneed.as<uint8_t>(), *have = b->xhave.as<uint8_t>();
		u32 *bounds = b->xmisc.as<u32>();                 // [0..6]
		unsigned int *n_retry = b->xmisc.as<unsigned int>() + 16, *n_unf = b->xmisc.as<unsigned int>() + 17, *n_heavy2 = b->xmisc.as<unsigned int>() + 26;
		int *sel_thresh = b->xmisc.as<int>() + 28;
		int n_in = n;
		rc = tier_threshold(b, "SSQ_HEAVY_TASKS", 32, sel_thresh);
		if (rc) return rc;
		CK(cudaMemsetAsync(b->xsel.p, 0, (size_t)(n + 1) * sizeof(SelState), b->st));
		CK(cudaMemsetAsync(b->xwide.p, 0, 2 * (nt + 1), b->st));
		CK(cudaMemsetAsync(need, 0, nt + 1, b->st)); CK(cudaMemsetAsync(have, 0, nt + 1, b->st));
		k_ext_prep<<<G, 256, 0, b->st>>>(b->idx->dev, b->opt, nt, b->tasks.as<Task>(), b->read_off.as<u64>(), b->intv_off.as<u64>(), b->seed_off.as<u64>(), b->outc.as<ChainRec>(),
		                                b->sorted.as<Seed>(), b->xinfo.as<ExtInfo>());
		const int lazy = getenv("SSQ_EXT_ALL") ? 0 : 1;
		const int force_round = getenv("SSQ_EXT_FORCE_ROUND") ? atoi(getenv("SSQ_EXT_FORCE_ROUND")) : 2; // from this round on an unfinished read gets all its remaining seeds extended
		if (lazy) k_need_first<<<(n + 255) / 256, 256, 0, b->st>>>(n, b->intv_off.as<u64>(), b->seed_off.as<u64>(), b->outc.as<ChainRec>(), b->sorted.as<Seed>(), b->n_kept.as<i32>(), b->task_off.as<u64>(), need);
		else CK(cudaMemsetAsync(need, 1, nt, b->st));
		b->launches += 3;
		static const int caps[6] = {32, 64, 96, 128, 160, 255};
		CK(cudaFuncSetAttribute(k_ext_run<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 131072 + 8192));
		CK(cudaFuncSetAttribute(k_ext_run<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 131072 + 8192));
		const size_t rsmem = (size_t)64 * (b->max_len + 2) * 4;
		CK(cudaFuncSetAttribute(k_ext_retry<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rsmem));
		CK(cudaFuncSetAttribute(k_ext_retry<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rsmem));
		const cudaEvent_t es0 = b->evx[0], es1 = b->evx[1];
		for (int round = 0;; ++round) {
			for (int dir = 0; dir < 2; ++dir) {
				size_t tb = 0;
				k_ext_keys<<<G, 256, 0, b->st>>>(dir, nt, b->xinfo.as<ExtInfo>(), need, have, b->xkey[0].as<u32>(), b->xidx[0].as<u32>());
				cub::DeviceRadixSort::SortPairs(0, tb, b->xkey[0].as<u32>(), b->xkey[1].as<u32>(), b->xidx[0].as<u32>(), b->xidx[1].as<u32>(), (int)nt, 0, 32, b->st);
				if (b->cubtmp.need(tb)) return SSQ_ENOMEM;
				CK(cub::DeviceRadixSort::SortPairs(b->cubtmp.p, tb, b->xkey[0].as<u32>(), b->xkey[1].as<u32>(), b->xidx[0].as<u32>(), b->xidx[1].as<u32>(), (int)nt, 0, 32, b->st));
				k_ext_bounds<<<1, 32, 0, b->st>>>(nt, b->xkey[1].as<u32>(), bounds);
				CK(cudaMemsetAsync(n_retry, 0, 4, b->st));
				u32 hb[8];
				CK(cudaMemcpyAsync(hb, bounds, 7 * 4, cudaMemcpyDeviceToHost, b->st));
				CK(cudaStreamSynchronize(b->st));
				b->launches += 4;
				for (int c = 5; c >= 0; --c) { // longest class first
					const u32 lo = hb[c], hi = hb[c + 1];
					if (hi <= lo) continue;
					const int threads = caps[c] > 160 ? 64 : 128;
					const size_t smem = (size_t)threads * (caps[c] + 2) * 4;
					const unsigned grid = (hi - lo + threads - 1) / threads;
					if (dir == 0)
						k_ext_run<0><<<grid, threads, smem, b->st>>>(b->idx->dev, b->opt, lo, hi, b->xidx[1].as<u32>(), b->tasks.as<Task>(), b->seq.as<uint8_t>(), b->read_off.as<u64>(),
						                                            b->xinfo.as<ExtInfo>(), b->cand.as<RegCand>(), b->xres[0].as<ExtRes>(), b->xretry.as<u32>(), n_retry, &b->misc.as<Misc>()->cnt);
					else
						k_ext_run<1><<<grid, threads, smem, b->st>>>(b->idx->dev, b->opt, lo, hi, b->xidx[1].as<u32>(), b->tasks.as<Task>(), b->seq.as<uint8_t>(), b->read_off.as<u64>(),
						                                            b->xinfo.as<ExtInfo>(), b->cand.as<RegCand>(), b->xres[1].as<ExtRes>(), b->xretry.as<u32>(), n_retry, &b->misc.as<Misc>()->cnt);
					++b->launches;
				}
				if (dir == 0) {
					k_ext_retry<0><<<b->n_sm * 2, 64, rsmem, b->st>>>(b->idx->dev, b->opt, b->xretry.as<u32>(), n_retry, b->tasks.as<Task>(), b->seq.as<uint8_t>(), b->read_off.as<u64>(),
					                                                 b->xinfo.as<ExtInfo>(), b->cand.as<RegCand>(), b->xres[0].as<ExtRes>(), wide_l, &b->misc.as<Misc>()->cnt);
					k_ext_left_fin<<<G, 256, 0, b->st>>>(b->opt, nt, b->xinfo.as<ExtInfo>(), b->xres[0].as<ExtRes>(), b->cand.as<RegCand>(), need, have);
				} else {
					k_ext_retry<1><<<b->n_sm * 2, 64, rsmem, b->st>>>(b->idx->dev, b->opt, b->xretry.as<u32>(), n_retry, b->tasks.as<Task>(), b->seq.as<uint8_t>(), b->read_off.as<u64>(),
					                                                 b->xinfo.as<ExtInfo>(), b->cand.as<RegCand>(), b->xres[1].as<ExtRes>(), wide_r, &b->misc.as<Misc>()->cnt);
					k_ext_right_fin<<<G, 256, 0, b->st>>>(b->opt, nt, b->tasks.as<Task>(), b->intv_off.as<u64>(), b->seed_off.as<u64>(), b->outc.as<ChainRec>(), b->sorted.as<Seed>(),
					                                     b->xinfo.as<ExtInfo>(), b->xres[1].as<ExtRes>(), wide_l, wide_r, b->cand.as<RegCand>(), need, have);
				}
				b->launches += 2;
			}
			// continue the selection for the reads that are not finished yet
			unsigned int h_unf = 0;
			CK(cudaMemsetAsync(n_unf, 0, 4, b->st));
			CK(cudaMemsetAsync(n_heavy2, 0, 4, b->st));
			CK(cudaMemsetAsync(&b->misc.as<Misc>()->work, 0, 4, b->st));
			CK(cudaEventRecord(es0, b->st));
			const u32 *list_in = round == 0 ? (const u32*)0 : b->xlist[(round - 1) & 1].as<u32>();
			u32 *list_out = b->xlist[round & 1].as<u32>();
			k_select<<<b->n_sm * 8, 128, 0, b->st>>>(b->opt, n_in, list_in, b->read_off.as<u64>(), b->intv_off.as<u64>(), b->seed_off.as<u64>(), b->outc.as<ChainRec>(), b->sorted.as<Seed>(),
			                                        b->n_kept.as<i32>(), b->task_off.as<u64>(), b->cand.as<RegCand>(), b->srt.as<u64>(), b->regs.as<RegCand>(), b->n_regs.as<u32>(),
			                                        have, need, b->xsel.as<SelState>(), round >= force_round, list_out, n_unf, &b->misc.as<Misc>()->work, sel_thresh, b->xheavy.as<u32>(), n_heavy2);
			CK(cudaMemsetAsync(&b->misc.as<Misc>()->work, 0, 4, b->st));
			k_select_heavy<<<b->n_sm * 8, 128, 0, b->st>>>(b->opt, b->read_off.as<u64>(), b->intv_off.as<u64>(), b->seed_off.as<u64>(), b->outc.as<ChainRec>(), b->sorted.as<Seed>(),
			                                              b->n_kept.as<i32>(), b->task_off.as<u64>(), b->cand.as<RegCand>(), b->srt.as<u64>(), b->srt2.as<u64>(), b->regs.as<RegCand>(), b->n_regs.as<u32>(),
			                                              have, need, b->xsel.as<SelState>(), round >= force_round, list_out, n_unf, &b->misc.as<Misc>()->work, b->xheavy.as<u32>(), n_heavy2);
			CK(cudaEventRecord(es1, b->st));
			++b->launches;
			++b->launches;
			CK(cudaGetLastError());
			CK(cudaMemcpyAsync(&h_unf, n_unf, 4, cudaMemcpyDeviceToHost, b->st));
			CK(cudaStreamSynchronize(b->st));
			{ float ms = 0.f; cudaEventElapsedTime(&ms, es0, es1); ms_sel += ms; }
			b->ext_rounds = round + 1;
			if (h_unf == 0) break;
			n_in = (int)h_unf;
			if (round > 8) { ssq_set_error("seed-extension rounds did not converge"); return SSQ_ECUDA; }
		}
	} else {
		CK(cudaMemsetAsync(b->n_regs.p, 0, (size_t)(n + 1) * 4, b->st));
	}
	b->select_ms = ms_sel;
	CK(cudaEventRecord(b->ev[4], b->st));
	return SSQ_OK;
}

static int run_upto(ssq_batch *b, int last_stage) // 0 smem, 1 sa, 2 chain, 3 extend+select
{
	int rc;
	b->launches = 0;
	CK(cudaEventRecord(b->ev[0], b->st));
	if ((rc = run_smem(b))) return rc;
	CK(cudaEventRecord(b->ev[1], b->st));
	if (last_stage >= 1 && (rc = run_sa(b))) return rc;
	CK(cudaEventRecord(b->ev[2], b->st));
	if (last_stage >= 2 && (rc = run_chain(b))) return rc;
	CK(cudaEventRecord(b->ev[3], b->st));
	CK(cudaEventRecord(b->ev[4], b->st));
	if (last_stage >= 3 && (rc = run_extend(b))) return rc;
	CK(cudaEventRecord(b->ev[5], b->st));
	return SSQ_OK;
}

extern "C" int ssq_batch_run(ssq_batch_t *b)
{
	int rc = ssq_use_device(b->idx->device);
	if (rc) return rc;
	return run_upto(b, 3);
}

static int finish_counters(ssq_batch *b)
{
	Misc hm;
	CK(cudaMemcpyAsync(&hm, b->misc.p, sizeof(Misc), cudaMemcpyDeviceToHost, b->st));
	CK(cudaStreamSynchronize(b->st));
	b->h_cnt = hm.cnt;
	for (int i = 0; i < 5; ++i) cudaEventElapsedTime(&b->stage_ms[i], b->ev[i], b->ev[i + 1]);
	b->stage_ms[3] -= b->select_ms; b->stage_ms[4] += b->select_ms; // the selection replays run inside the extension rounds
	return SSQ_OK;
}

extern "C" uint64_t ssq_batch_counter(const ssq_batch_t *b_, int what)
{
	ssq_batch *b = (ssq_batch*)b_;
	if (finish_counters(b)) return 0;
	switch (what) {
	case 0: return b->h_cnt.occ_smem; case 1: return b->h_cnt.occ_sa; case 2: return b->h_cnt.sa_reads; case 3: return b->h_cnt.sw_calls;
	case 4: return b->h_cnt.sw_cells; case 5: return b->h_cnt.sw_bytes; case 6: return (uint64_t)b->launches; case 7: return b->n_seeds; case 8: return b->n_regs_total;
	case 9: return b->n_intv; case 10: return b->n_tasks; case 11: return (uint64_t)b->ext_rounds;
	case 12: case 13: case 14: case 15: case 16: return b->h_cnt.dbg[what - 12];
	case 23: return b->h_cnt.dbg[6]; // rank blocks dereferenced by k_smem_p3 (part of counter 0)
	case 25: return (b->h_cnt.dbg[9] - b->h_cnt.dbg[8]) + (b->h_cnt.dbg[11] - b->h_cnt.dbg[10]); // rank blocks dereferenced by the two backward-sweep launches (split seeding)
	case 26: { float m1 = 0.f, m2 = 0.f; if (cudaEventElapsedTime(&m1, b->evb[0], b->evb[1]) != cudaSuccess || cudaEventElapsedTime(&m2, b->evb[2], b->evb[3]) != cudaSuccess) { cudaGetLastError(); return 0; } return (uint64_t)((m1 + m2) * 1000.f); } // their duration, microseconds
	case 24: { float ms = 0.f; if (cudaEventElapsedTime(&ms, b->evs[0], b->evs[1]) != cudaSuccess) { cudaGetLastError(); return 0; } return (uint64_t)(ms * 1000.f); } // k_smem_m alone, microseconds
	case 22: { float ms = 0.f; cudaEventElapsedTime(&ms, b->evc[3], b->evc[2]); return (uint64_t)(ms * 1000.f); } // the big-shared-memory tier alone
	case 17: case 18: { float ms = 0.f; cudaEventElapsedTime(&ms, b->evc[what - 17], b->evc[what - 16]); return (uint64_t)(ms * 1000.f); } // chaining tiers, microseconds
	case 19: case 20: case 21: { u32 v = 0; cudaMemcpy(&v, b->xmisc.as<u32>() + (what == 19 ? 24 : what == 20 ? 27 : 25), 4, cudaMemcpyDeviceToHost); return v; } // reads in the warp tier; the cut; reads passed on to the big-shared-memory tier
	}
	return 0;
}

extern "C" float ssq_batch_stage_ms(const ssq_batch_t *b_, int stage)
{
	ssq_batch *b = (ssq_batch*)b_;
	if (stage < 0 || stage > 4 || finish_counters(b)) return -1.f;
	return b->stage_ms[stage];
}

extern "C" int ssq_batch_fetch(ssq_batch_t *b, ssq_alnreg_t *out, uint64_t out_cap, uint64_t *out_off, uint64_t *needed)
{
	const int n = b->n_reads;
	int rc = ssq_use_device(b->idx->device);
	if (rc) return rc;
	if (n == 0) { if (out_off) out_off[0] = 0; if (needed) *needed = 0; return SSQ_OK; }
	if (b->srt.need((size_t)(n + 2) * 8)) return SSQ_ENOMEM; // temp for widened counts (selection is finished by now)
	k_widen_u32<<<(n + 255) / 256, 256, 0, b->st>>>((u64)n, b->n_regs.as<u32>(), b->srt.as<u64>());
	if ((rc = scan_u64(b, b->srt.as<u64>(), b->reg_off.as<u64>(), (size_t)n + 1))) return rc;
	CK(cudaMemcpyAsync(&b->n_regs_total, b->reg_off.as<u64>() + n, 8, cudaMemcpyDeviceToHost, b->st));
	CK(cudaStreamSynchronize(b->st));
	if (needed) *needed = b->n_regs_total;
	if (out_off) CK(cudaMemcpyAsync(out_off, b->reg_off.p, (size_t)(n + 1) * 8, cudaMemcpyDeviceToHost, b->st));
	if (b->n_regs_total > out_cap || !out) { CK(cudaStreamSynchronize(b->st)); return b->n_regs_total > out_cap ? SSQ_ECAP : SSQ_OK; }
	if (b->out.need((b->n_regs_total + 1) * sizeof(ssq_alnreg_t))) return SSQ_ENOMEM;
	k_gather_regs<<<(n + 255) / 256, 256, 0, b->st>>>(n, b->task_off.as<u64>(), b->reg_off.as<u64>(), b->n_regs.as<u32>(), b->regs.as<RegCand>(), b->out.as<ssq_alnreg_t>());
	CK(cudaGetLastError());
	CK(cudaMemcpyAsync(out, b->out.p, b->n_regs_total * sizeof(ssq_alnreg_t), cudaMemcpyDeviceToHost, b->st));
	CK(cudaStreamSynchronize(b->st));
	return SSQ_OK;
}

extern "C" int ssq_align_batch(const ssq_index_t *idx, const ssq_opts_t *opt, int n_reads, const uint8_t *seq, const uint64_t *read_off,
                               int stage, ssq_alnreg_t *out, uint64_t out_cap, uint64_t *out_off, uint64_t *needed)
{
	ssq_batch_t *b = 0;
	if (stage != 0) { ssq_set_error("ssq_align_batch: only stage 0 (regions out of seed extension) is implemented"); return SSQ_EINVAL; }
	int rc = ssq_batch_create(idx, opt, n_reads, seq, read_off, &b);
	if (rc) return rc;
	rc = ssq_batch_run(b);
	if (!rc) rc = ssq_batch_fetch(b, out, out_cap, out_off, needed);
	ssq_batch_free(b);
	return rc;
}

// ------------------------------------------------------------ kernel-level C-ABI entry points ----
extern "C" int ssq_smem_batch(const ssq_index_t *idx, const ssq_opts_t *opt, int n_reads, const uint8_t *seq, const uint64_t *read_off,
                              ssq_smem_t *out, uint64_t out_cap, uint64_t *out_off, uint64_t *needed)
{
	ssq_batch_t *b = 0;
	int rc = ssq_batch_create(idx, opt, n_reads, seq, read_off, &b);
	if (rc) return rc;
	rc = run_upto(b, 0);
	if (!rc && n_reads > 0) {
		const int n = n_reads;
		do {
			if (b->srt.need((size_t)(n + 2) * 8) || b->reg_off.need((size_t)(n + 2) * 8)) { rc = SSQ_ENOMEM; break; }
			k_widen_i32<<<(n + 255) / 256, 256, 0, b->st>>>(n, b->intv_cnt.as<i32>(), b->srt.as<u64>());
			if ((rc = scan_u64(b, b->srt.as<u64>(), b->reg_off.as<u64>(), (size_t)n + 1))) break;
			if (needed) *needed = b->n_intv;
			if (cudaMemcpyAsync(out_off, b->reg_off.p, (size_t)(n + 1) * 8, cudaMemcpyDeviceToHost, b->st) != cudaSuccess) { rc = SSQ_ECUDA; break; }
			if (b->n_intv > out_cap) { cudaStreamSynchronize(b->st); rc = SSQ_ECAP; break; }
			if (b->out.need((b->n_intv + 1) * sizeof(ssq_smem_t))) { rc = SSQ_ENOMEM; break; }
			k_gather_intv<<<(n + 255) / 256, 256, 0, b->st>>>(n, b->intv_off.as<u64>(), b->intv_cnt.as<i32>(), b->reg_off.as<u64>(), b->pool.as<Intv>(), b->out.as<ssq_smem_t>());
			if (cudaMemcpyAsync(out, b->out.p, b->n_intv * sizeof(ssq_smem_t), cudaMemcpyDeviceToHost, b->st) != cudaSuccess || cudaStreamSynchronize(b->st) != cudaSuccess) {
				ssq_set_error("copy-back failed: %s", cudaGetErrorString(cudaGetLastError())); rc = SSQ_ECUDA;
			}
		} while (0);
	} else if (!rc) { out_off[0] = 0; if (needed) *needed = 0; }
	ssq_batch_free(b);
	return rc;
}

extern "C" int ssq_chain_batch(const ssq_index_t *idx, const ssq_opts_t *opt, int n_reads, const uint8_t *seq, const uint64_t *read_off,
                               ssq_seed_t *seeds, uint64_t seed_cap, uint64_t *chain_seed_off, uint64_t chain_cap, uint64_t *read_chain_off,
                               uint64_t *n_chains, uint64_t *n_seeds)
{
	ssq_batch_t *b = 0;
	int rc = ssq_batch_create(idx, opt, n_reads, seq, read_off, &b);
	if (rc) return rc;
	rc = run_upto(b, 2);
	const int n = n_reads;
	if (!rc && n > 0) {
		do {
			DBuf cdst, sdst, tmp, d_seeds, d_cso;
			u64 nc = 0, ns = 0;
			if (cdst.need((size_t)(n + 2) * 8) || sdst.need((size_t)(n + 2) * 8) || tmp.need((size_t)(n + 2) * 8)) { rc = SSQ_ENOMEM; break; }
			k_widen_i32<<<(n + 255) / 256, 256, 0, b->st>>>(n, b->n_kept.as<i32>(), tmp.as<u64>());
			if ((rc = scan_u64(b, tmp.as<u64>(), cdst.as<u64>(), (size_t)n + 1))) break;
			k_widen_u32<<<(n + 255) / 256, 256, 0, b->st>>>((u64)n, b->n_kseeds.as<u32>(), tmp.as<u64>());
			if ((rc = scan_u64(b, tmp.as<u64>(), sdst.as<u64>(), (size_t)n + 1))) break;
			cudaMemcpyAsync(&nc, cdst.as<u64>() + n, 8, cudaMemcpyDeviceToHost, b->st);
			cudaMemcpyAsync(&ns, sdst.as<u64>() + n, 8, cudaMemcpyDeviceToHost, b->st);
			cudaMemcpyAsync(read_chain_off, cdst.p, (size_t)(n + 1) * 8, cudaMemcpyDeviceToHost, b->st);
			if (cudaStreamSynchronize(b->st) != cudaSuccess) { rc = SSQ_ECUDA; break; }
			if (n_chains) *n_chains = nc;
			if (n_seeds) *n_seeds = ns;
			if (nc > chain_cap || ns > seed_cap) { rc = SSQ_ECAP; cdst.release(); sdst.release(); tmp.release(); break; }
			if (d_seeds.need((ns + 1) * sizeof(ssq_seed_t)) || d_cso.need((nc + 2) * 8)) { rc = SSQ_ENOMEM; break; }
			k_gather_chains<<<(n + 255) / 256, 256, 0, b->st>>>(n, b->intv_off.as<u64>(), b->intv_cnt.as<i32>(), b->seed_off.as<u64>(), b->outc.as<ChainRec>(), b->sorted.as<Seed>(),
			                                                   b->n_kept.as<i32>(), cdst.as<u64>(), sdst.as<u64>(), d_seeds.as<ssq_seed_t>(), d_cso.as<u64>());
			cudaMemcpyAsync(seeds, d_seeds.p, ns * sizeof(ssq_seed_t), cudaMemcpyDeviceToHost, b->st);
			cudaMemcpyAsync(chain_seed_off, d_cso.p, nc * 8, cudaMemcpyDeviceToHost, b->st);
			if (cudaStreamSynchronize(b->st) != cudaSuccess) { ssq_set_error("chain copy-back: %s", cudaGetErrorString(cudaGetLastError())); rc = SSQ_ECUDA; }
			chain_seed_off[nc] = ns;
			cdst.release(); sdst.release(); tmp.release(); d_seeds.release(); d_cso.release();
		} while (0);
	} else if (!rc) { read_chain_off[0] = 0; chain_seed_off[0] = 0; if (n_chains) *n_chains = 0; if (n_seeds) *n_seeds = 0; }
	ssq_batch_free(b);
	return rc;
}

extern "C" int ssq_sa_lookup_batch(const ssq_index_t *idx, uint64_t n, const uint64_t *rows, uint64_t *pos)
{
	int rc = ssq_use_device(idx->device);
	if (rc) return rc;
	if (n == 0) return SSQ_OK;
	DBuf in, out;
	if (in.need(n * 8) || out.need(n * 8)) return SSQ_ENOMEM;
	CK(cudaMemcpy(in.p, rows, n * 8, cudaMemcpyHostToDevice));
	k_sa_rows<<<(unsigned)((n + 255) / 256), 256>>>(idx->dev, n, in.as<u64>(), out.as<u64>());
	CK(cudaGetLastError());
	CK(cudaMemcpy(pos, out.p, n * 8, cudaMemcpyDeviceToHost));
	in.release(); out.release();
	return SSQ_OK;
}

extern "C" int ssq_sw_extend_batch(const ssq_opts_t *opt, int device, uint64_t n, const ssq_sw_task_t *tasks,
                                   const uint8_t *qbuf, uint64_t qbuf_len, const uint8_t *tbuf, uint64_t tbuf_len, ssq_sw_result_t *out)
{
	int rc = ssq_use_device(device);
	if (rc) return rc;
	if (n == 0) return SSQ_OK;
	int qmax = 0;
	for (u64 i = 0; i < n; ++i) {
		if (tasks[i].qlen < 1 || tasks[i].qlen > SSQ_MAX_READ_LEN || tasks[i].h0 < 1 || tasks[i].q_off + tasks[i].qlen > qbuf_len || tasks[i].t_off + tasks[i].tlen > tbuf_len) {
			ssq_set_error("ssq_sw_extend_batch: task %llu out of range", (unsigned long long)i); return SSQ_EINVAL;
		}
		if ((long long)tasks[i].h0 + (long long)tasks[i].qlen * opt->a > 65535) { // the DP row keeps H and E in 16 bits each (sw_extend_impl)
			ssq_set_error("ssq_sw_extend_batch: task %llu: h0 + qlen * a = %lld exceeds 65535, the largest score the DP row holds", (unsigned long long)i,
			              (long long)tasks[i].h0 + (long long)tasks[i].qlen * opt->a);
			return SSQ_EINVAL;
		}
		if (tasks[i].qlen > qmax) qmax = tasks[i].qlen;
	}
	DBuf dt, dq, dtb, dout;
	if (dt.need(n * sizeof(ssq_sw_task_t)) || dq.need(qbuf_len + 16) || dtb.need(tbuf_len + 16) || dout.need(n * sizeof(ssq_sw_result_t))) return SSQ_ENOMEM;
	CK(cudaMemcpy(dt.p, tasks, n * sizeof(ssq_sw_task_t), cudaMemcpyHostToDevice));
	CK(cudaMemcpy(dq.p, qbuf, qbuf_len, cudaMemcpyHostToDevice));
	CK(cudaMemcpy(dtb.p, tbuf, tbuf_len, cudaMemcpyHostToDevice));
	const int threads = 64;
	const size_t smem = (size_t)threads * (qmax + 2) * 4;
	CK(cudaFuncSetAttribute(k_sw_tasks, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
	k_sw_tasks<<<(unsigned)((n + threads - 1) / threads), threads, smem>>>(*opt, n, dt.as<ssq_sw_task_t>(), dq.as<uint8_t>(), dtb.as<uint8_t>(), dout.as<ssq_sw_result_t>());
	CK(cudaGetLastError());
	CK(cudaMemcpy(out, dout.p, n * sizeof(ssq_sw_result_t), cudaMemcpyDeviceToHost));
	dt.release(); dq.release(); dtb.release(); dout.release();
	return SSQ_OK;
}

extern "C" int ssq_dupmark_batch(int device, uint64_t n, const ssq_dupsig_t *sig, uint8_t *is_dup)
{
	int rc = ssq_use_device(device);
	if (rc) return rc;
	if (n == 0) return SSQ_OK;
	if (n >= 0x7fffffffull) { ssq_set_error("ssq_dupmark_batch: more than 2^31-1 pairs in one call (the sort takes a 32-bit item count)"); return SSQ_EINVAL; }
	DBuf dsig, k1, k2, k1g, ka, idx_a, idx_b, tmp, dd;
	if (dsig.need(n * sizeof(ssq_dupsig_t)) || k1.need(n * 8) || k2.need(n * 8) || k1g.need(n * 8) || ka.need(n * 8) || idx_a.need(n * 4) || idx_b.need(n * 4) || dd.need(n)) return SSQ_ENOMEM;
	CK(cudaMemcpy(dsig.p, sig, n * sizeof(ssq_dupsig_t), cudaMemcpyHostToDevice));
	const unsigned g = (unsigned)((n + 255) / 256);
	k_dup_keys<<<g, 256>>>(n, dsig.as<ssq_dupsig_t>(), k1.as<u64>(), k2.as<u64>(), idx_a.as<u32>());
	size_t tb = 0;
	cub::DeviceRadixSort::SortPairs(0, tb, k2.as<u64>(), ka.as<u64>(), idx_a.as<u32>(), idx_b.as<u32>(), (int)n);
	if (tmp.need(tb)) return SSQ_ENOMEM;
	CK(cub::DeviceRadixSort::SortPairs(tmp.p, tb, k2.as<u64>(), ka.as<u64>(), idx_a.as<u32>(), idx_b.as<u32>(), (int)n)); // stable, by key2
	k_dup_gather<<<g, 256>>>(n, idx_b.as<u32>(), k1.as<u64>(), k1g.as<u64>());
	CK(cub::DeviceRadixSort::SortPairs(tmp.p, tb, k1g.as<u64>(), ka.as<u64>(), idx_b.as<u32>(), idx_a.as<u32>(), (int)n)); // stable, by key1
	k_dup_mark<<<g, 256>>>(n, idx_a.as<u32>(), ka.as<u64>(), k2.as<u64>(), dsig.as<ssq_dupsig_t>(), dd.as<uint8_t>());
	CK(cudaGetLastError());
	CK(cudaMemcpy(is_dup, dd.p, n, cudaMemcpyDeviceToHost));
	DBuf *all[] = {&dsig, &k1, &k2, &k1g, &ka, &idx_a, &idx_b, &tmp, &dd};
	for (size_t i = 0; i < 9; ++i) all[i]->release();
	return SSQ_OK;
}

// --------------------------------------------------------------------------- streaming dup-set ----
// First-seen-wins across a stream of batches (what `$SAMBLASTER` needs: its input does not fit one call).  The set of
// signatures seen so far is kept on the device as two parallel arrays sorted by (key1, key2); a batch is (1) marked within
// itself by the two-pass stable sort above, (2) its survivors are looked up in the set by binary search, (3) the new ones
// are appended and the set is re-sorted (two stable LSD passes).
struct __align__(16) P128 { u64 a, b; };
struct P128Lt { __host__ __device__ bool operator()(const P128 &x, const P128 &y) const { return x.a < y.a || (x.a == y.a && x.b < y.b); } };
struct ssq_dupset {
	int device; u64 n, cap; P128 *keys, *alt; // every signature seen so far, sorted by (key1, key2); alt: the other half of the double buffer the merge writes into
	DBuf m1, m2, k1g, ka, idx_a, idx_b, tmp, dnew, cnt, s128, sflag, n128; /* scratch kept across calls */
	std::mutex mu; std::condition_variable cv; long long turn; // batches of one run mark in batch order even when several host threads drive them
};

__global__ void k_dupset_lookup(u64 n, const ssq_dupsig_t *__restrict__ sig, const u64 *__restrict__ key1, const u64 *__restrict__ key2, uint8_t *is_dup,
                                const u64 *__restrict__ s1, const u64 *__restrict__ s2, u64 sn, uint8_t *is_new)
{
	u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	uint8_t nw = 0;
	if (sig[i].valid && !is_dup[i]) {
		const u64 a = key1[i], b = key2[i];
		u64 lo = 0, hi = sn;
		while (lo < hi) { const u64 mid = (lo + hi) >> 1; if (s1[mid] < a || (s1[mid] == a && s2[mid] < b)) lo = mid + 1; else hi = mid; }
		if (lo < sn && s1[lo] == a && s2[lo] == b) is_dup[i] = 1; else nw = 1;
	}
	is_new[i] = nw;
}

extern "C" int ssq_dupset_create(int device, ssq_dupset_t **out)
{
	int rc = ssq_use_device(device);
	if (rc) return rc;
	ssq_dupset *s = new ssq_dupset();
	s->device = device; s->n = s->cap = 0; s->keys = s->alt = 0; s->turn = 0;
	*out = s;
	return SSQ_OK;
}
extern "C" void ssq_dupset_free(ssq_dupset_t *s) { if (!s) return; cudaFree(s->keys); cudaFree(s->alt); delete s; }
extern "C" uint64_t ssq_dupset_size(const ssq_dupset_t *s) { return s ? s->n : 0; }

__global__ void k_dupset_lookup_keys(u64 n, const uint8_t *__restrict__ valid, const u64 *__restrict__ key1, const u64 *__restrict__ key2, uint8_t *is_dup,
                                     const P128 *__restrict__ set, u64 sn, uint8_t *is_new)
{
	u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	uint8_t nw = 0;
	if (valid[i] && !is_dup[i]) {
		const u64 a = key1[i], b = key2[i];
		u64 lo = 0, hi = sn;
		while (lo < hi) { const u64 mid = (lo + hi) >> 1; const P128 v = set[mid]; if (v.a < a || (v.a == a && v.b < b)) lo = mid + 1; else hi = mid; }
		if (lo < sn) { const P128 v = set[lo]; if (v.a == a && v.b == b) is_dup[i] = 1; else nw = 1; } else nw = 1;
	}
	is_new[i] = nw;
}
// the chunk's items in sorted order (idx = the order the two stable sort passes produced): their keys as one 128-bit word and whether they are new
__global__ void k_dup_sorted_new(u64 n, const u32 *__restrict__ idx, const u64 *__restrict__ key1s, const u64 *__restrict__ key2, const uint8_t *__restrict__ is_new, P128 *out, uint8_t *flag)
{
	u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const u32 me = idx[i];
	P128 v; v.a = key1s[i]; v.b = key2[me];
	out[i] = v; flag[i] = is_new[me];
}
__global__ void k_dup_sig_keys(u64 n, const ssq_dupsig_t *__restrict__ sig, u64 *key1, u64 *key2, uint8_t *valid)
{
	u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	key1[i] = sig[i].pos1 << 1 | (sig[i].strand1 & 1); key2[i] = sig[i].pos2 << 1 | (sig[i].strand2 & 1); valid[i] = sig[i].valid ? 1 : 0;
}
__global__ void k_dup_iota(u64 n, u32 *idx);
__global__ void k_dup_mask(u64 n, const uint8_t *__restrict__ valid, const u64 *__restrict__ k1, const u64 *__restrict__ k2, u64 *m1, u64 *m2);
__global__ void k_dup_mark_keys(u64 n, const u32 *__restrict__ idx, const u64 *__restrict__ key1s, const u64 *__restrict__ key2, const uint8_t *__restrict__ valid, uint8_t *is_dup);

extern "C" int ssq_dupset_reset(ssq_dupset_t *set) { if (!set) return SSQ_EINVAL; std::lock_guard<std::mutex> g(set->mu); set->n = 0; set->turn = 0; set->cv.notify_all(); return SSQ_OK; }
// "first seen wins" is defined by input order: when batches are driven concurrently (one host thread and stream per batch), each
// waits here until every earlier batch (turn = 0, 1, 2, ... since the last reset) has gone through the set
extern "C" void ssq_dupset_wait_turn(ssq_dupset_t *set, long long turn) { std::unique_lock<std::mutex> l(set->mu); set->cv.wait(l, [&] { return set->turn >= turn; }); }
extern "C" void ssq_dupset_end_turn(ssq_dupset_t *set, long long turn) { std::lock_guard<std::mutex> g(set->mu); if (set->turn == turn) set->turn = turn + 1; set->cv.notify_all(); }

// Device-pointer form (the fused `bwa mem | samblaster` path, ssq_pipe.cu): key1/key2 = (5' position << 1 | strand) of the
// canonically ordered ends, element order = input order.  Marks duplicates within the chunk (two stable radix-sort passes +
// adjacent-equal test), then against the sorted set of every earlier chunk (binary search), then absorbs the new signatures.
extern "C" int ssq_dupset_mark_dev(ssq_dupset_t *set, uint64_t n, const uint64_t *d_k1, const uint64_t *d_k2, const uint8_t *d_valid, uint8_t *d_is_dup, void *stream_)
{
	if (!set) return SSQ_EINVAL;
	int rc = ssq_use_device(set->device);
	if (rc) return rc;
	if (n == 0) return SSQ_OK;
	if (n >= 0x7fffffffull) { ssq_set_error("ssq_dupset_mark: more than 2^31-1 pairs in one call"); return SSQ_EINVAL; }
	cudaStream_t st = (cudaStream_t)stream_;
	DBuf &m1 = set->m1, &m2 = set->m2, &k1g = set->k1g, &ka = set->ka, &idx_a = set->idx_a, &idx_b = set->idx_b, &tmp = set->tmp, &dnew = set->dnew, &cnt = set->cnt;
	if (m1.need(n * 8) || m2.need(n * 8) || k1g.need(n * 8) || ka.need(n * 8) || idx_a.need(n * 4) || idx_b.need(n * 4) || dnew.need(n) || cnt.need(16) || set->s128.need(n * 16) || set->sflag.need(n) ||
	    set->n128.need(n * 16)) return SSQ_ENOMEM;
	const unsigned g = (unsigned)((n + 255) / 256);
	const u64 grown = set->n + n;
	if (grown >= 0x7fffffffull) { ssq_set_error("ssq_dupset: more than 2^31-1 distinct signatures"); return SSQ_ECAP; }
	size_t tb = 0, tb2 = 0;
	cub::DeviceRadixSort::SortPairs(0, tb, m2.as<u64>(), ka.as<u64>(), idx_a.as<u32>(), idx_b.as<u32>(), (int)n, 0, 64, st);
	cub::DeviceSelect::Flagged(0, tb2, set->s128.as<P128>(), set->sflag.as<uint8_t>(), set->n128.as<P128>(), cnt.as<u64>(), (int)n, st);
	if (tb2 > tb) tb = tb2;
	cub::DeviceMerge::MergeKeys(0, tb2, (const P128*)0, (int)set->n, (const P128*)0, (int)n, (P128*)0, P128Lt(), st);
	if (tb2 > tb) tb = tb2;
	if (tmp.need(tb)) return SSQ_ENOMEM;
	k_dup_mask<<<g, 256, 0, st>>>(n, d_valid, d_k1, d_k2, m1.as<u64>(), m2.as<u64>());
	k_dup_iota<<<g, 256, 0, st>>>(n, idx_a.as<u32>());
	CK(cub::DeviceRadixSort::SortPairs(tmp.p, tb, m2.as<u64>(), ka.as<u64>(), idx_a.as<u32>(), idx_b.as<u32>(), (int)n, 0, 64, st)); // stable, by key2
	k_dup_gather<<<g, 256, 0, st>>>(n, idx_b.as<u32>(), m1.as<u64>(), k1g.as<u64>());
	CK(cub::DeviceRadixSort::SortPairs(tmp.p, tb, k1g.as<u64>(), ka.as<u64>(), idx_b.as<u32>(), idx_a.as<u32>(), (int)n, 0, 64, st)); // stable, by key1: now sorted by (key1, key2), input order inside equal keys
	k_dup_mark_keys<<<g, 256, 0, st>>>(n, idx_a.as<u32>(), ka.as<u64>(), m2.as<u64>(), d_valid, d_is_dup);
	k_dupset_lookup_keys<<<g, 256, 0, st>>>(n, d_valid, d_k1, d_k2, d_is_dup, set->keys, set->n, dnew.as<uint8_t>());
	// absorb the new signatures: they are already in sorted order inside the chunk, so the set grows by ONE merge (16 B/key read +
	// written), not by a re-sort of everything seen so far
	k_dup_sorted_new<<<g, 256, 0, st>>>(n, idx_a.as<u32>(), ka.as<u64>(), m2.as<u64>(), dnew.as<uint8_t>(), set->s128.as<P128>(), set->sflag.as<uint8_t>());
	CK(cudaGetLastError());
	u64 n_new = 0;
	CK(cub::DeviceSelect::Flagged(tmp.p, tb, set->s128.as<P128>(), set->sflag.as<uint8_t>(), set->n128.as<P128>(), cnt.as<u64>(), (int)n, st));
	CK(cudaMemcpyAsync(&n_new, cnt.p, 8, cudaMemcpyDeviceToHost, st));
	CK(cudaStreamSynchronize(st));
	if (n_new) {
		const u64 total = set->n + n_new;
		if (total > set->cap) { // grow both halves of the double buffer, keeping the content
			const u64 ncap = total + total / 2 + 1024;
			P128 *a = 0, *b = 0;
			CK(cudaMalloc(&a, ncap * sizeof(P128))); CK(cudaMalloc(&b, ncap * sizeof(P128)));
			if (set->n) CK(cudaMemcpyAsync(a, set->keys, set->n * sizeof(P128), cudaMemcpyDeviceToDevice, st));
			CK(cudaStreamSynchronize(st));
			cudaFree(set->keys); cudaFree(set->alt);
			set->keys = a; set->alt = b; set->cap = ncap;
		}
		CK(cub::DeviceMerge::MergeKeys(tmp.p, tb, (const P128*)set->keys, (int)set->n, (const P128*)set->n128.as<P128>(), (int)n_new, set->alt, P128Lt(), st));
		P128 *t = set->keys; set->keys = set->alt; set->alt = t;
		set->n = total;
	}
	return SSQ_OK;
}

extern "C" int ssq_dupset_mark(ssq_dupset_t *set, uint64_t n, const ssq_dupsig_t *sig, uint8_t *is_dup)
{
	if (!set) return SSQ_EINVAL;
	int rc = ssq_use_device(set->device);
	if (rc) return rc;
	if (n == 0) return SSQ_OK;
	if (n >= 0x7fffffffull) { ssq_set_error("ssq_dupset_mark: more than 2^31-1 pairs in one call"); return SSQ_EINVAL; }
	DBuf dsig, k1, k2, va, dd;
	if (dsig.need(n * sizeof(ssq_dupsig_t)) || k1.need(n * 8) || k2.need(n * 8) || va.need(n) || dd.need(n)) return SSQ_ENOMEM;
	CK(cudaMemcpy(dsig.p, sig, n * sizeof(ssq_dupsig_t), cudaMemcpyHostToDevice));
	k_dup_sig_keys<<<(unsigned)((n + 255) / 256), 256>>>(n, dsig.as<ssq_dupsig_t>(), k1.as<u64>(), k2.as<u64>(), va.as<uint8_t>());
	CK(cudaGetLastError());
	CK(cudaDeviceSynchronize());
	if ((rc = ssq_dupset_mark_dev(set, n, k1.as<u64>(), k2.as<u64>(), va.as<uint8_t>(), dd.as<uint8_t>(), 0))) return rc;
	CK(cudaMemcpy(is_dup, dd.p, n, cudaMemcpyDeviceToHost));
	return SSQ_OK;
}

// ------------------------------------------------------------- device-resident dup-marking ----
// keys already in HBM (e.g. received through an NCCL all-to-all): key1/key2 = (pos << 1 | strand) of the canonically
// ordered ends, valid[i] = 0 for pairs that can never be duplicates; elements are taken in array order (= first-seen order).
__global__ void k_dup_iota(u64 n, u32 *idx) { u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; if (i < n) idx[i] = (u32)i; }
__global__ void k_dup_mask(u64 n, const uint8_t *__restrict__ valid, const u64 *__restrict__ k1, const u64 *__restrict__ k2, u64 *m1, u64 *m2)
{
	u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
	if (i < n) { m1[i] = valid[i] ? k1[i] : ~0ull; m2[i] = valid[i] ? k2[i] : ~0ull; }
}
__global__ void k_dup_mark_keys(u64 n, const u32 *__restrict__ idx, const u64 *__restrict__ key1s, const u64 *__restrict__ key2, const uint8_t *__restrict__ valid, uint8_t *is_dup)
{
	u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const u32 me = idx[i];
	uint8_t d = 0;
	if (i > 0 && valid[me]) { const u32 pv = idx[i - 1]; d = valid[pv] && key1s[i] == key1s[i - 1] && key2[me] == key2[pv]; }
	is_dup[me] = d;
}

extern "C" int ssq_dupmark_keys_dev(int device, uint64_t n, const uint64_t *d_key1, const uint64_t *d_key2, const uint8_t *d_valid, uint8_t *d_is_dup, void *stream_)
{
	int rc = ssq_use_device(device);
	if (rc) return rc;
	if (n == 0) return SSQ_OK;
	if (n >= 0x7fffffffull) { ssq_set_error("ssq_dupmark_keys_dev: more than 2^31-1 pairs in one call (the sort takes a 32-bit item count)"); return SSQ_EINVAL; }
	cudaStream_t st = (cudaStream_t)stream_;
	DBuf m1, m2, k1g, ka, idx_a, idx_b, tmp;
	if (m1.need(n * 8) || m2.need(n * 8) || k1g.need(n * 8) || ka.need(n * 8) || idx_a.need(n * 4) || idx_b.need(n * 4)) return SSQ_ENOMEM;
	const unsigned g = (unsigned)((n + 255) / 256);
	k_dup_mask<<<g, 256, 0, st>>>(n, d_valid, d_key1, d_key2, m1.as<u64>(), m2.as<u64>());
	k_dup_iota<<<g, 256, 0, st>>>(n, idx_a.as<u32>());
	size_t tb = 0;
	cub::DeviceRadixSort::SortPairs(0, tb, m2.as<u64>(), ka.as<u64>(), idx_a.as<u32>(), idx_b.as<u32>(), (int)n, 0, 64, st);
	if (tmp.need(tb)) return SSQ_ENOMEM;
	CK(cub::DeviceRadixSort::SortPairs(tmp.p, tb, m2.as<u64>(), ka.as<u64>(), idx_a.as<u32>(), idx_b.as<u32>(), (int)n, 0, 64, st));
	k_dup_gather<<<g, 256, 0, st>>>(n, idx_b.as<u32>(), m1.as<u64>(), k1g.as<u64>());
	CK(cub::DeviceRadixSort::SortPairs(tmp.p, tb, k1g.as<u64>(), ka.as<u64>(), idx_b.as<u32>(), idx_a.as<u32>(), (int)n, 0, 64, st));
	k_dup_mark_keys<<<g, 256, 0, st>>>(n, idx_a.as<u32>(), ka.as<u64>(), m2.as<u64>(), d_valid, d_is_dup);
	CK(cudaGetLastError());
	CK(cudaStreamSynchronize(st));
	return SSQ_OK;
}
