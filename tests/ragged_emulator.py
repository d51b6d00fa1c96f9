"""Test-only model of a ragged run (include/signalops.h `sigops_plan_run_ragged`) on top of tests/plan_emulator.py.

It follows the runtime's rules: one plan (the field-wise maximum of the elements'), instances sorted longest first
(caller order when the plan draws device noise) and cut into waves, every stage of a wave computed over the prefix its
longest instance needs (rounded up to 16 frames within the plan's), rows zero past each instance's valid frames
(inputs on arrival, temps after their producer), each sum of squares taken over the instance's valid frames and scaled
by d0 / (N_i * C), and only the valid frames copied out.  Temps start out NaN, as a stale workspace would, so that a
missing zero tail shows in the results.
"""
import numpy as np

from plan_emulator import NP, Emulator


def _round16(n):
    return (n + 15) // 16 * 16


class RaggedEmulator(Emulator):
    def slot_d0(self):
        d = {}
        for I in self.instrs:
            if I[1] == 7 and 1 <= I[0] <= 5:
                d[I[4]] = I[10]
        return d

    def has_randn(self):
        return any(I[1] == 9 and (1 <= I[0] <= 5 or I[0] == 15) for I in self.instrs)

    def run_ragged(self, inputs, out_frames, temp_frames, wave=2):
        """inputs: [ninst][n_in] arrays of each instance's own frames; out_frames: [ninst] root frames; temp_frames:
        [ninst][n_tmp].  Returns [ninst] lists of outputs."""
        ninst = len(inputs)
        nb = len(self.bufdesc)
        valid = np.zeros((ninst, nb), dtype=np.int64)
        for i in range(ninst):
            valid[i, :self.n_in] = [len(a) for a in inputs[i]]
            valid[i, self.n_in:self.n_in + self.n_tmp] = temp_frames[i]
            valid[i, self.n_in + self.n_tmp:] = out_frames[i]
        order = list(range(ninst))
        if not self.has_randn():
            order.sort(key=lambda i: -int(out_frames[i]))
        results = [None] * ninst
        for w0 in range(0, ninst, wave):
            members = order[w0:w0 + wave]
            vmax = valid[members].max(axis=0)
            prefix = [min(self.bufdesc[st[1]][0], _round16(int(vmax[st[1]]))) for st in self.stages]
            for pos, i in enumerate(members, w0):
                # (the instance index a kernel sees is the position in the run, which picks the noise stream)
                results[i] = self._run_instance(inputs[i], valid[i], prefix, pos)
        return results

    def _run_instance(self, inputs, valid, prefix, inst):
        self.inst = inst
        d0 = self.slot_d0()
        self.bufs = []
        for k, (n, c, dt) in enumerate(self.bufdesc):
            fill = np.nan if NP[dt] != np.int64 else np.iinfo(np.int64).max // 3
            b = np.full((n, c), fill, dtype=NP[dt])
            if k < self.n_in:
                a = np.asarray(inputs[k]).reshape(len(inputs[k]), c)
                b[:len(a)] = a
                b[len(a):] = 0                                      # zero tail after the copy-in
            self.bufs.append(b)
        self.scalars = np.zeros(max(1, self.n_scal))
        for si, st in enumerate(self.stages):
            (kind, out_buf, slot, p0, npc, in0, inl, ep0, epl, nch, n_in, n_out, *rest) = st
            n = prefix[si]
            ob = self.bufs[out_buf]

            def store(idx, c, v):
                ob[idx, c] = v.astype(ob.dtype)

            if kind == 1:
                for (lo, ln, c0, cc, ps, pl) in self.pieces[p0:p0 + npc]:
                    idx = np.arange(lo, max(lo, min(lo + ln, n)))
                    for c in range(c0, c0 + cc):
                        store(idx, c, self.run_prog(ps, pl, idx, c))
            elif n > 0:
                m_in = n if kind == 2 else n_in                     # a FIR reads its whole (zero-tailed) input
                cut = (kind, out_buf, slot, p0, npc, in0, inl, ep0, epl, nch, m_in, n, *rest)
                for c in range(nch):
                    x = self.run_prog(in0, inl, np.arange(m_in), c) if m_in else np.zeros(0)
                    if kind == 2:
                        from scipy import signal as sps
                        M, ctab, gain = rest[0], rest[1], rest[2]
                        coef = self.tables[ctab].reshape(M, 5)
                        sos = np.column_stack([coef[:, :3], np.ones(M), coef[:, 3:]])
                        y = sps.sosfilt(sos, x) * gain
                    else:
                        y = self.fir(cut, x)
                    idx = np.arange(n)
                    store(idx, c, self.run_prog(ep0, epl, idx, c, y) if epl else y)
            v = int(valid[out_buf])
            if slot >= 0:
                s = float(np.sum(ob[:v].astype(np.float64) ** 2))
                self.scalars[slot] = s * d0.get(slot, 0.0) / (v * ob.shape[1]) if v else 0.0
            if out_buf < self.n_in + self.n_tmp:
                ob[v:] = 0                                          # zero tail after the producer
        return [self.bufs[k][:valid[k]] for k in range(self.n_in + self.n_tmp, len(self.bufdesc))]
