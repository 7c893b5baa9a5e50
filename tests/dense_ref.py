"""Dense float64 reference of gen_dist for the independent-genotype and called-genotype paths (no product code here).

Restated from oracle/ngsdist_oracle.c, not from the CUDA sources.  With independent genotypes the sum of gen_dist is a
sum of matrix products, so a whole matrix at the benchmark's shapes is a few float64 GEMMs (cuBLAS through torch on a
CUDA device, or the CPU):

  A = M o P (the planes g = 0, 1, 2; M the presence mask under --pairwise_del, all ones otherwise),
  B = (S (M o P))_g, i.e. B[j, s, g1] = sum_g2 score[g1][g2] A[j, s, g2],
  num_b = A_b B_b^T and cnt_b = M_b M_b^T over the sites of bootstrap block b (K = 3 x the block's sites),

so entry (i, j), i < j, has row individual i take g1 as in gen_dist_pair.  Replicate r adds c_{r,b} num_b and
c_{r,b} cnt_b over the blocks, with c_{0,b} = 1 for every site (the n_sites % block_size tail included) and c_{r,b} for
r >= 1 the multiplicities of rnd_map_data (oracle.Taus), over the persistently truncated n_sites.  `finish` is the tail of
gen_dist: tot_sites, models 0, 1 and 2, a zero diagonal and a mirrored upper triangle.

On the called path with --pairwise_del every operand entry is 0 or 1 and every score 0, 1/2 or 1, so num is exact.
"""
import math

import numpy as np
import torch

import oracle

NGSD_INF = 1e15     # ngsdist_oracle.c NGSD_INF
EPS = 1e-5          # ngsdist_oracle.c NGSD_EPS
KNIFE = 1e-11       # a miss_data3 difference this close to EPS, or a threshold comparison this close, is a knife edge


def boot_counts(seed, n_sites, block_size, n_rep):
    """Block multiplicities of replicates 1 .. n_rep (ngsDist.cpp:235-238 through oracle.Taus): [n_rep][n_sites // bs]."""
    rng = oracle.Taus(seed)
    out = []
    for _ in range(n_rep):
        n_sites -= n_sites % block_size
        nb = n_sites // block_size
        sm = rng.boot_map(nb, block_size)
        out.append(np.bincount((sm[::block_size] // np.uint64(block_size)).astype(np.int64), minlength=nb))
    return np.array(out, dtype=np.float64).reshape(n_rep, -1)


def frontend(raw, call_geno=False, N_thresh=0.0, call_thresh=0.0):
    """frontend_one for the binary reader in normal scale, on raw [m][n][3] -> P [n][m][3] (same device).
    Also returns a boolean [n][m] of knife-edge triples: a call rule comparison (tie or threshold) within KNIFE."""
    L = torch.log(raw.permute(1, 0, 2))
    L = torch.where(L == -math.inf, torch.full_like(L, -NGSD_INF), L)
    l0, l1, l2 = L.unbind(-1)
    M = torch.where(l1 >= l0, l1, l0)
    M = torch.where(l2 >= M, l2, M)
    s = torch.exp(l0 - M) + torch.exp(l1 - M)
    s = s + torch.exp(l2 - M)
    norm = torch.where(M == -math.inf, M, torch.log(s) + M)       # logsum3
    L = L - norm.unsqueeze(-1)                                    # post_prob3
    if torch.isnan(L).any():
        raise ValueError("NaN found! Is the file format correct?")
    knife = torch.zeros(L.shape[:2], dtype=torch.bool, device=L.device)
    if call_geno:                                                 # call_geno3
        if N_thresh > call_thresh:
            raise ValueError("missing data threshold must be smaller than calling genotype threshold!")
        l0, l1, l2 = L.unbind(-1)
        mx_pos = torch.zeros_like(l0, dtype=torch.int64)
        mx = l0
        mx_pos = torch.where(l1 > mx, 1, mx_pos); mx = torch.where(l1 > mx, l1, mx)
        mx_pos = torch.where(l2 > mx, 2, mx_pos); mx = torch.where(l2 > mx, l2, mx)
        mn = torch.minimum(torch.minimum(l0, l1), l2)
        max_pp = torch.where(mn == mx, torch.full_like(mx, -1.0), torch.exp(mx))
        srt = L.sort(-1).values
        knife |= (srt[..., 1] == srt[..., 2]) & (mn != mx)        # two equal maxima: the first one is called
        for t in (N_thresh, call_thresh):
            knife |= (max_pp - t).abs() <= KNIFE
        L = torch.where((max_pp < N_thresh).unsqueeze(-1), torch.full_like(L, math.log(1.0 / 3)), L)
        onehot = torch.full_like(L, -NGSD_INF).scatter_(-1, mx_pos.unsqueeze(-1), 0.0)
        L = torch.where((max_pp >= call_thresh).unsqueeze(-1), onehot, L)
    return torch.exp(L), knife


def present(P):
    """Not miss_data3, [n][m] bool; and the triples whose outcome a difference within KNIFE of EPS could flip."""
    d01 = (P[..., 0] - P[..., 1]).abs()
    d12 = (P[..., 1] - P[..., 2]).abs()
    knife = (((d01 - EPS).abs() <= KNIFE) & (d12 < EPS + KNIFE)) | (((d12 - EPS).abs() <= KNIFE) & (d01 < EPS + KNIFE))
    return ~((d01 < EPS) & (d12 < EPS)), knife


class DenseRef:
    """Streaming accumulator: add() raw chunks of sites in any order, then finish().

    counts: [n_rep][n_sites // block_size] multiplicities of the bootstrap replicates (boot_counts), or None for
    replicate 0 alone.  Replicate 0 is always result 0."""

    def __init__(self, n_ind, n_sites, *, score=None, pairwise_del=False, call_geno=False, N_thresh=0.0, call_thresh=0.0,
                 block_size=1, counts=None, device="cpu"):
        self.n, self.n_sites, self.bs = n_ind, n_sites, block_size
        self.pdel, self.call = pairwise_del, (call_geno, N_thresh, call_thresh)
        self.device = torch.device(device)
        S = oracle.DEFAULT_SCORE if score is None else np.asarray(score, dtype=np.float64).reshape(9)
        self.ST = torch.tensor(S.reshape(3, 3).T.copy(), dtype=torch.float64, device=self.device)
        self.score_span = max(S.max(), 0.0) - min(S.min(), 0.0)   # the most one site of one pair can move num
        nwb = -(-n_sites // block_size)                      # weight blocks: the last may be partial
        W = np.zeros((1 + (0 if counts is None else len(counts)), nwb))
        W[0] = 1.0
        if counts is not None and len(counts):
            W[1:, :counts.shape[1]] = counts
        self.W = W
        self.R = W.shape[0]
        self.num = torch.zeros((self.R, n_ind * n_ind), dtype=torch.float64, device=self.device)
        self.cnt = torch.zeros((self.R, n_ind * n_ind), dtype=torch.float64, device=self.device)
        self.knife = []          # (individual, site, raw triple) of every knife-edge triple met

    def add(self, raw, site0):
        """raw: [m][n_ind][3] float64 tensor (binary layout, normal scale) of sites site0 .. site0 + m."""
        raw = raw.to(self.device)
        m = raw.shape[0]
        P, kn = frontend(raw, *self.call)
        if self.pdel:
            Mk, kn2 = present(P)
            kn |= kn2
            A = P * Mk.unsqueeze(-1).to(P.dtype)
        else:
            Mk, A = None, P
        del P
        for i, s in kn.nonzero().tolist():
            self.knife.append((i, site0 + s, raw[s, i].tolist()))
        B = A @ self.ST                                       # B[j, s, g1] = sum_g2 score[g1][g2] A[j, s, g2]
        if self.R == 1:
            pieces = [(0, m, 0)]
        else:                                                 # cut at bootstrap block boundaries
            pieces, s = [], 0
            while s < m:
                b = (site0 + s) // self.bs
                e = min(m, (b + 1) * self.bs - site0)
                pieces.append((s, e, b))
                s = e
        for s, e, b in pieces:
            w = self.W[:, b]
            rows = np.nonzero(w)[0]
            if len(rows) == 0:
                continue
            a = A[:, s:e].reshape(self.n, -1)
            num_b = (a @ B[:, s:e].reshape(self.n, -1).T).view(-1)
            if self.pdel:
                mk = Mk[:, s:e].to(torch.float64)
                cnt_b = (mk @ mk.T).view(-1)
            for r in rows:
                self.num[r].add_(num_b, alpha=float(w[r]))
                if self.pdel:
                    self.cnt[r].add_(cnt_b, alpha=float(w[r]))
                else:
                    self.cnt[r].add_(float(w[r] * (e - s)))

    def knife_sites(self, r):
        """{individual: {site: (multiplicity in replicate r, raw triple)}} of the knife-edge triples replicate r uses.
        One such site moves cnt of a pair by at most its multiplicity, and num by at most that times score_span."""
        out = {}
        for i, site, triple in self.knife:
            w = float(self.W[r, site // self.bs])
            if w:
                out.setdefault(i, {})[site] = (w, triple)
        return out

    def finish(self, r, tot_sites=0, evol_model=1):
        """Replicate r: dict(dist, num, cnt) of n x n float64 tensors (cnt holds integers), as gen_dist returns them."""
        n = self.n
        num = torch.triu(self.num[r].view(n, n), 1)
        cnt = torch.triu(self.cnt[r].view(n, n), 1)
        d = num / (cnt if tot_sites == 0 else torch.full_like(cnt, float(tot_sites)))
        if evol_model == 1:
            d = -torch.log(1 - d)
        elif evol_model == 2:
            d = -torch.log(1 - (d * 4 / 3)) * 3 / 4
        elif evol_model != 0:
            raise ValueError("invalid evolutionary model specified!")
        d = torch.triu(d, 1)
        return dict(dist=d + d.T, num=num + num.T, cnt=cnt + cnt.T)
