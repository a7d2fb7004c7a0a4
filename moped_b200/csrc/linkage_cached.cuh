// linkage_cached.cuh — hierarchicalCluster of moped3d's CLUSTER_LINKAGE_CPU (moped3d/libmoped/src/cluster/CLUSTER_LINKAGE_CPU.hpp:414-531,
// average linkage) with a CACHED MAXIMUM PER ROW: the same merge sequence as the reference — its scan-order tie rule (first
// maximum of the double loop), the stale column of the merged-away cluster and the list element its erase-then-++ skips —
// but a merge costs O(n) plus the rows whose cached maximum was invalidated instead of an O(n^2) scan of all live pairs
// (profiles/launches_r1k_linkage_summary.md: that scan is 98 % of the stage). The algorithm is the one modelled and checked
// against the oracle in scripts/linkage_cached_model.py.
//
// Invariant per live list position a (list L of cluster ids, ascending; posOf = inverse):
//     best[L[a]] = max over later positions b of D[L[a]][L[b]],  arg[L[a]] = the id at the SMALLEST such b   (strict > in scan order)
// NaN similarities (duplicate matches) never win a strict >, so the max skips them like the reference's scan: best is never NaN
// (-1 when a row has no finite entry left), and every repair below keeps it so.
//
// Written for a block of W threads as a sequence of phases (`blk.each(f)`: __syncthreads(); f(tid); __syncthreads(); on the
// device, a loop over the threads on the host), so that tests/cpp/linkage_host.cpp can compile this very source with g++ and
// compare it with the oracle on a machine without a GPU (both thread orders). Not a CPU path of the product.
#pragma once

#include <stdint.h>
#include <stddef.h>

#include "simt_phases.cuh"

#define LKX_FN PHX_FN
#define LKX_MEM PHX_MEM

namespace lkx {

template <int W> using Block = phx::BlockTeam<W>;    // the CTA as a team (simt_phases.cuh)

struct State {
	int n;
	float *D;                 // n x n working similarities
	int *L, *posOf;           // live cluster ids in list order, and the position of an id
	float *best; int *arg;    // cached row maximum (by cluster id) and the id of its column
	int *lists, *sz;          // members of cluster i: lists[i*n .. i*n+sz[i])
	float *tmp, *oldcol;      // n each
	int *tmpi;                // n
	float *s_val; int *s_idx; // W each (shared memory on the device)
	int *ctl;                 // 16 control words (shared memory on the device)
};
enum { C_NL = 0, C_REMOVE, C_STOP, C_P1, C_P2, C_SU, C_SR, C_BESTPOS, C_R };

// best / arg of the row at list position pos, scanned by ONE thread in list order
LKX_FN void recompute_row(const State &s, int pos, int nL) {
	const int i = s.L[pos];
	float b = -1.f; int a = -1;
	const float *row = s.D + (size_t)i * s.n;
	for (int q = pos + 1; q < nL; q++) {
		const float v = row[s.L[q]];
		if (v > b) { b = v; a = s.L[q]; }
	}
	s.best[i] = b; s.arg[i] = a;
}

// block-wide (max value, ties -> smallest index) of the candidates every thread left in s_val / s_idx; result in slot 0
template <int W>
LKX_FN void reduce_max_first(const Block<W> &blk, const State &s) {
	for (int o = W / 2; o > 0; o >>= 1)
		blk.each([&](int t) {
			if (t < o) {
				const float v2 = s.s_val[t + o]; const int i2 = s.s_idx[t + o];
				if (v2 > s.s_val[t] || (v2 == s.s_val[t] && i2 < s.s_idx[t])) { s.s_val[t] = v2; s.s_idx[t] = i2; }
			}
		});
}

// K: n x n similarities (the lower triangle j >= i is read, like distances[j*N+i] = distances[i*N+j] = K->getProb(i, j), :434-439).
// Outputs: clusters with more than min_pts members in index order (CSR). Returns nothing; *out_count = number of clusters.
template <int W>
LKX_FN void agglomerate_average(const Block<W> &blk, const State &s, const float *K, float cutoff, int min_pts, int *out_count,
                                int *out_offsets, int *out_members) {
	const int n = s.n;
	blk.each([&](int t) {
		for (size_t k = t; k < (size_t)n * n; k += W) {
			const int i = (int)(k / n), j = (int)(k % n);
			s.D[k] = j >= i ? K[(size_t)j * n + i] : K[(size_t)i * n + j];
		}
		for (int i = t; i < n; i += W) { s.L[i] = i; s.posOf[i] = i; s.lists[(size_t)i * n] = i; s.sz[i] = 1; }
		if (t == 0) { s.ctl[C_NL] = n; s.ctl[C_REMOVE] = -1; s.ctl[C_STOP] = 0; }
	});
	blk.each([&](int t) {
		for (int pos = t; pos < n; pos += W) recompute_row(s, pos, n);
	});
	for (;;) {
		const int nL = s.ctl[C_NL], remove = s.ctl[C_REMOVE];
		const int r = remove >= 0 ? s.posOf[remove] : -1;
		// the pass maximum: first row in list order (not r, not r+1: erase-then-++ skips it) whose cached maximum is the largest
		blk.each([&](int t) {
			float mx = -1.f; int bp = 0x7fffffff;
			for (int a = t; a < nL; a += W) {
				if (r >= 0 && (a == r || a == r + 1)) continue;
				const float v = s.best[s.L[a]];
				if (v > mx) { mx = v; bp = a; }
			}
			s.s_val[t] = mx; s.s_idx[t] = bp;
		});
		reduce_max_first(blk, s);
		blk.each([&](int t) {
			if (t == 0) {
				const int bp = s.s_idx[0];
				s.ctl[C_BESTPOS] = bp;
				s.ctl[C_P1] = bp < nL ? s.L[bp] : -1;
				s.ctl[C_P2] = bp < nL ? s.arg[s.L[bp]] : -1;      // the pair is fixed here: the stale column may be the winner
			}
		});
		const float mx = s.s_val[0];
		int nLn = nL;
		if (r >= 0) {                                           // validIndices.erase(position r)
			const int gone = s.L[r];
			blk.each([&](int t) {
				for (int k = r + t; k < nL - 1; k += W) s.tmpi[k] = s.L[k + 1];
			});
			blk.each([&](int t) {
				for (int k = r + t; k < nL - 1; k += W) { s.L[k] = s.tmpi[k]; s.posOf[s.tmpi[k]] = k; }
				if (t == 0) { s.ctl[C_NL] = nL - 1; s.posOf[gone] = -1; }      // a stale winner may name it again: then nothing is erased
			});
			nLn = nL - 1;
			blk.each([&](int t) {                                // rows before it that pointed at it lose their maximum
				for (int pos = t; pos < r; pos += W)
					if (s.arg[s.L[pos]] == gone) recompute_row(s, pos, nLn);
			});
		}
		const int p1 = s.ctl[C_P1], p2 = s.ctl[C_P2];
		if (mx < cutoff || p1 < 0 || p2 < 0) break;
		blk.each([&](int t) {
			if (t == 0) {
				s.ctl[C_SU] = s.sz[p1]; s.ctl[C_SR] = s.sz[p2];
				int *l1 = s.lists + (size_t)p1 * n, *l2 = s.lists + (size_t)p2 * n;      // the second cluster is appended back to front (:480-483)
				while (s.sz[p2] != 0) l1[s.sz[p1]++] = l2[--s.sz[p2]];
				s.ctl[C_REMOVE] = p2;
			}
		});
		const int sU = s.ctl[C_SU], sR = s.ctl[C_SR];
		// row / column of the merged cluster (:489-512): every i reads the OLD (p1, i) and (p2, i)
		blk.each([&](int t) {
			for (int i = t; i < n; i += W) {
				s.oldcol[i] = s.D[(size_t)i * n + p1];
				s.tmp[i] = (float)((1.0 / (sU + sR)) * (sU * s.D[(size_t)p1 * n + i] + sR * s.D[(size_t)p2 * n + i]));
			}
		});
		blk.each([&](int t) {
			for (int i = t; i < n; i += W) { s.D[(size_t)p1 * n + i] = s.tmp[i]; s.D[(size_t)i * n + p1] = s.tmp[i]; }
		});
		// the merged cluster's own row: block-wide scan of its later positions
		const int pos1 = s.posOf[p1];
		blk.each([&](int t) {
			float b = -1.f; int bq = 0x7fffffff;
			const float *row = s.D + (size_t)p1 * n;
			for (int q = pos1 + 1 + t; q < nLn; q += W) {
				const float v = row[s.L[q]];
				if (v > b) { b = v; bq = q; }
			}
			s.s_val[t] = b; s.s_idx[t] = bq;
		});
		reduce_max_first(blk, s);
		// rows before it: their entry in column p1 changed
		blk.each([&](int t) {
			if (t == 0) { s.best[p1] = s.s_val[0]; s.arg[p1] = s.s_idx[0] < nLn ? s.L[s.s_idx[0]] : -1; }
			for (int pos = t; pos < pos1; pos += W) {
				const int i = s.L[pos];
				const float v = s.D[(size_t)i * n + p1];
				if (s.arg[i] == p1) {
					// NaN (0/0 of the 3-D filter at duplicate matches) never wins a compare: rescan instead of caching it
					if (!(v >= s.oldcol[i])) recompute_row(s, pos, nLn);
					else s.best[i] = v;
				} else if (v > s.best[i] || (v == s.best[i] && s.arg[i] >= 0 && s.posOf[s.arg[i]] > pos1)) {
					s.best[i] = v; s.arg[i] = p1;
				}
			}
		});
	}
	blk.each([&](int t) {
		if (t == 0) {                                           // clusters with more than MinPts members, in index order (:519-529)
			int nc = 0, k = 0;
			out_offsets[0] = 0;
			for (int i = 0; i < n; i++)
				if (s.sz[i] > min_pts) {
					const int *l = s.lists + (size_t)i * n;
					for (int a = 0; a < s.sz[i]; a++) out_members[k++] = l[a];
					out_offsets[++nc] = k;
				}
			*out_count = nc;
		}
	});
}

} // namespace lkx
