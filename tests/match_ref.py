"""Sequential restatement of the match model (cz_model_set_match, include/candlezip_b200.h), for the tests: per segment, a table of the most
recent position of every context key, the verify-and-length rule, per-bucket counts of tries and hits, and the interval list the coder
lanes code.  Nothing here is shared with the CUDA code."""
import numpy as np

HB, NB, TOTAL = 18, 16, 1 << 30
NONE = 2 ** 32 - 1


def context_key(ctx):
    """key over the K symbols before a position, oldest first"""
    h = 0x811C9DC5
    for x in ctx:
        h = ((h ^ int(x)) * 0x01000193) & 0xFFFFFFFF
    return ((h * 0x9E3779B1) & 0xFFFFFFFF) >> (32 - HB)


def weight(hits, tries):
    p16 = ((2 * hits + 1) << 16) // (2 * tries + 2)
    return min(max(p16, 1), 65535) << 14


def segment_predictions(t, K):
    """per position of one segment's symbols t: (pred or NONE, W or 0, bucket or -1)"""
    assert 1 <= K <= 16
    t = [int(x) for x in t]
    n = len(t)
    pred, w, bucket = [NONE] * n, [0] * n, [-1] * n
    table, tries, hits = {}, [0] * NB, [0] * NB
    for i in range(n):
        if i >= K:
            key = context_key(t[i - K:i])
            j = table.get(key)
            table[key] = i
            if j is not None:
                length = 0
                while length < K + NB - 1 and j - 1 - length >= 0 and t[j - 1 - length] == t[i - 1 - length]:
                    length += 1
                if length >= K:
                    b = length - K
                    pred[i], w[i], bucket[i] = t[j], weight(hits[b], tries[b]), b
        if pred[i] != NONE:
            tries[bucket[i]] += 1
            hits[bucket[i]] += t[i] == pred[i]
    return pred, w, bucket


def predictions(ids, seg_start, K):
    """segment_predictions over every segment of a call: (pred, W) uint32 arrays by global coded index"""
    ids = np.asarray(ids, np.uint32)
    pred, w = np.full(ids.shape[0], NONE, np.uint32), np.zeros(ids.shape[0], np.uint32)
    for a, b in zip(seg_start[:-1], seg_start[1:]):
        p, ww, _ = segment_predictions(ids[int(a):int(b)], K)
        pred[int(a):int(b)], w[int(a):int(b)] = p, ww
    return pred, w


def interval_list(ids, pred, w, c_lo, c_hi):
    """the intervals one segment's lane codes: per token, the flag when it has a prediction, then the model's interval unless a hit"""
    out = []
    for x, p, ww, lo, hi in zip(ids, pred, w, c_lo, c_hi):
        if p != NONE:
            if x == p:
                out.append((0, int(ww)))
                continue
            out.append((int(ww), TOTAL))
        out.append((int(lo), int(hi)))
    return out
