"""Executable specification of FM-index extract (include/bwts_b200.h, bwts_b200_fm_extract_*): a numpy restatement
of the GPU path (bijective-bwt_b200/csrc/fm.cuh, k_fm_isa / k_fm_seg_scan / k_fm_extract) on top of
fm_oracle.FmModel -- the inverse table of the samples derived block by block from the marks, the directory and the
samples, the 64-bit segment offsets, and the LF walk of each segment from the row of its end.  Nothing in the
product imports this module."""
import numpy as np

import fm_oracle


class ExtractModel:
    def __init__(self, model: fm_oracle.FmModel):
        self.m = model
        self.sh = model.sample.bit_length() - 1
        assert 1 << self.sh == model.sample
        self.isa = self.derive_isa()

    def derive_isa(self):
        """k_fm_isa: per 256-row block b, its marked rows in order take the ranks dir[b], dir[b] + 1, ...; the row r
        with value v = samples[rank] sets isa[v >> sh] = r + 1; isa[ceil(n / sample)] = 0, the $ row"""
        m, n = self.m, self.m.n
        nsamp = (n + m.sample - 1) >> self.sh
        isa = np.full(nsamp + 1, -1, dtype=np.int64)
        isa[nsamp] = 0
        for b in range((n + 255) // 256):
            rows = b * 256 + np.nonzero(m.marks[b * 256:(b + 1) * 256])[0]
            ranks = int(m.dir[b]) + np.arange(len(rows))
            isa[m.samples[ranks] >> self.sh] = rows + 1
        assert (isa >= 0).all()
        return isa

    def segment_offsets(self, a, b):
        """k_fm_seg_scan: exclusive 64-bit prefix of ceil(b / s) - floor(a / s) (0 for an empty range)"""
        a, b = np.asarray(a, np.int64), np.asarray(b, np.int64)
        cnt = np.where(a < b, ((b - 1) >> self.sh) - (a >> self.sh) + 1, 0)
        return np.concatenate([[0], np.cumsum(cnt)]).astype(np.int64)

    def walk(self, q, first, end, out, base):
        """segment q from the row of its end down to position `first`; positions below `end` are written"""
        m = self.m
        p = min((q + 1) << self.sh, m.n)
        i = int(self.isa[q + 1])
        steps = 0
        while True:
            assert i != m.primary
            c = int(m.U[i - (i > m.primary)])
            p -= 1
            steps += 1
            if p < end:
                out[base + p] = c
            if p == first:
                break
            i = int(m.C[c]) + m.occ(c, i)
        assert steps <= m.sample
        return steps

    def extract(self, a, b):
        """the bytes T[a_0:b_0] . T[a_1:b_1] . ..., segment by segment in the order of the GPU's half-warps"""
        a, b = np.asarray(a, np.int64), np.asarray(b, np.int64)
        offs = np.concatenate([[0], np.cumsum(b - a)]).astype(np.int64)
        segs = self.segment_offsets(a, b)
        out = np.full(int(offs[-1]), -1, dtype=np.int64)
        for g in range(int(segs[-1])):
            k = int(np.searchsorted(segs, g, side="right")) - 1     # largest k with segs[k] <= g
            ak, bk = int(a[k]), int(b[k])
            q = (ak >> self.sh) + g - int(segs[k])
            self.walk(q, max(ak, q << self.sh), bk, out, int(offs[k]) - ak)
        assert (out >= 0).all()
        return out.astype(np.uint8), offs
