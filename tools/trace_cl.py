#!/usr/bin/env python
"""Summarise a BWGR_TRACE file of the CLUSTERED pipelined sweep: [cta][block][32] = 16 globaltimer (ns) + 16 clock64 stamps.
CTA 8c = solver of cluster c (8 h received, 9 corrected, 10 solved, 11 published; 4 = comm warps: grid sum ready),
CTA 8c + r = its workers (0 step received, 1 DL written, 2 U issued, 3 u_done, 4 U-epilogue done, 5 G issued, 6 g_done, 7 partial sent
= added to the grid-sum words of h).
Traces of the kernel before the grid-sum words (partials summed per cluster, the cluster sums exchanged through an L2 ring) also
carry, on the solver, 5 = the seven partials of the cluster arrived, 6 = the cluster's sum stored, 12 = the last cluster's word
seen; the leg "last partial sent -> grid sum ready" is then split at those stamps."""
import sys
import numpy as np
raw = np.fromfile(sys.argv[1], dtype=np.int64)
G, nb, K, D = raw[:4]
t = raw[4:].reshape(G, nb, K).astype(np.float64)
lo, hi = 50, min(350, nb - 4)
b = np.arange(lo, hi)
c = b + 1 + D
S = t[0]
ck = 16
print("grid", G, "blocks", nb, "D", D)
print("solver period: %.0f ns (globaltimer), %.0f cycles" % (np.median(np.diff(S[lo:hi, 11])), np.median(np.diff(S[lo:hi, ck + 11]))))
print("solver cycles: grid sum ready(comm) -> h read %d | h read -> corrected %d | corrected -> solved %d | solved -> published %d | published -> next grid sum ready %d" % (
    np.median(S[b, ck + 8] - S[b, ck + 4]), np.median(S[b, ck + 9] - S[b, ck + 8]), np.median(S[b, ck + 10] - S[b, ck + 9]),
    np.median(S[b, ck + 11] - S[b, ck + 10]), np.median(S[b + 1, ck + 4] - S[b, ck + 11])))
for wk in (1, 7, 8 * (G // 16) + 3, G - 1):
    x = t[wk]
    f = lambda k1, b1, k0, b0: np.median(x[b1, ck + k1] - x[b0, ck + k0])
    print("worker cta %3d cycles: step recv->DL %d | DL->U issued %d | U issued->u_done %d | u_done->U-epi %d | U-epi->G issued %d | G issued->g_done %d | g_done->partial sent %d | sent->next step recv %d" % (
        wk, f(1, b, 0, b), f(2, b, 1, b), f(3, b, 2, b), f(4, b, 3, b), f(5, b, 4, b), f(6, c, 5, b), f(7, c, 6, c), f(0, b + 1, 7, c)))
# cross-CTA (globaltimer, coarse): solver 0 published -> its workers received; workers sent -> solver grid sum ready
w = t[1:8]
print("cluster 0 (ns, globaltimer): published -> step received by its workers: med %.0f max %.0f" % (np.median(w[:, b, 0] - S[b, 11][None, :]), np.median((w[:, b, 0] - S[b, 11][None, :]).max(0))))
allw = np.array([t[i] for i in range(G) if i % 8 != 0])
last_sent = allw[:, c, 7].max(0)
print("last partial sent by ANY worker -> grid sum ready at solver 0: med %.0f ns ; last partial of cluster 0 -> ready: %.0f ns" % (
    np.median(S[c, 4] - last_sent), np.median(S[c, 4] - w[:, c, 7].max(0))))
sol = t[0::8]
print("grid sum ready across solvers (ns): spread med %.0f ; published spread med %.0f" % (np.median(sol[:, b, 4].max(0) - sol[:, b, 4].min(0)), np.median(sol[:, b, 11].max(0) - sol[:, b, 11].min(0))))
first_recv = allw[:, b, 0].min(0); last_recv = allw[:, b, 0].max(0)
print("step received: first worker - solver0 published %.0f ns, last worker %.0f ns" % (np.median(first_recv - S[b, 11]), np.median(last_recv - S[b, 11])))
sent = allw[:, c, 7]
print("partial sent (block c=b+1+D) relative to step received (block b): med %.0f ns, slowest worker med %.0f ns" % (np.median(sent - allw[:, b, 0]), np.median((sent - allw[:, b, 0]).max(0))))
# the leg "last partial sent -> grid sum ready", split (older kernel only).  Cycles on solver 0's SM; ns (globaltimer) across SMs
if bool((S[b, 5] != 0).all()):
    has12 = bool((S[b, 12] != 0).all())
    print("solver 0 cycles: partials in -> cluster sum stored %d | stored -> %s %d" % (
        np.median(S[c, ck + 6] - S[c, ck + 5]),
        "last cluster word seen %d | seen -> grid sum ready" % np.median(S[c, ck + 12] - S[c, ck + 6]) if has12 else "grid sum ready",
        np.median(S[c, ck + 4] - S[c, ck + (12 if has12 else 6)])))
    last_stored = sol[:, c, 6].max(0)
    print("last partial sent by ANY worker -> last cluster's partials in (any solver): med %.0f ns ; -> last cluster sum stored (any solver): med %.0f ns ; "
          "last cluster sum stored -> grid sum ready at solver 0: med %.0f ns" % (
              np.median(sol[:, c, 5].max(0) - last_sent), np.median(last_stored - last_sent), np.median(S[c, 4] - last_stored)))
