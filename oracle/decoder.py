"""TEST INFRASTRUCTURE: CPU restatement of the reference's Viterbi decoder, the host counterpart of
the GPU search in pocketkaldi_b200/csrc/decoder.cu. tests/test_oracle.py pins it to the reference's
own decodes of the toy model (tests/golden/toy_decode_ref.txt)."""

import numpy as np


def host_viterbi(graph, tid2pdf, loglik, beam=16.0):
    """CPU restatement of the reference decoder (Decoder::Decode, src/decoder.cc:39-339) over
    scaled log-likelihoods [T][pdfs], in its arithmetic: float token costs, arc totals in double,
    weight cutoff float(best + beam), next cutoff the least kept emitting total + beam, epsilon
    closure under float(next cutoff), a token replaced only by a strictly lower cost, and the best
    final token's weight with its final weight added twice. Returns (word ids, weight)."""
    num_states, start, finals, arcs = graph
    out = [[] for _ in range(num_states)]
    for src, dst, il, ol, w in arcs:
        out[src].append((dst, il, ol, float(np.float32(w))))
    f32 = lambda x: float(np.float32(x))

    def close(toks, cutoff):
        queue = list(toks)
        while queue:
            s = queue.pop()
            cost, words = toks[s]
            for dst, il, ol, w in out[s]:
                if il != 0 or cost + w > cutoff:
                    continue
                c = f32(cost + w)
                if dst not in toks or c < toks[dst][0]:
                    toks[dst] = (c, words + (ol,) if ol else words)
                    queue.append(dst)

    toks = {start: (0.0, ())}
    close(toks, np.inf)
    for row in loglik:
        weight_cutoff = f32(min(c for c, _ in toks.values()) + beam)
        cand = [(cost + w - float(row[tid2pdf[il]]), dst, ol, words)
                for s, (cost, words) in toks.items() if cost <= weight_cutoff
                for dst, il, ol, w in out[s] if il != 0]
        if not cand:
            return [], 0.0
        next_cutoff = min(c[0] for c in cand) + beam
        new = {}
        for total, dst, ol, words in cand:
            if total > next_cutoff:
                continue
            c = f32(total)
            if dst not in new or c < new[dst][0]:
                new[dst] = (c, words + (ol,) if ol else words)
        close(new, f32(next_cutoff))
        toks = new
    ends = [(f32(c + finals[s]), s, words) for s, (c, words) in toks.items() if s in finals]
    if not ends:
        return [], 0.0
    c, s, words = min(ends)
    return list(words), f32(c + finals[s])


def host_decode(oracle, graph, tid2pdf, layers, prior, g, pcms):
    """The reference CLI's path on the host: fbank -> CMVN -> decodable (prob_scale 0.1) through the
    C restatement (oracle/pk_oracle.c), then host_viterbi. Returns [(word ids, weight / frames)]."""
    res = []
    for pcm in pcms:
        ft = oracle.cmvn(oracle.fbank(pcm.astype(np.float32)), g)
        ll = oracle.decodable(ft, layers, prior, 5, 5, 0.1)
        ids, w = host_viterbi(graph, tid2pdf, ll)
        res.append((ids, w / max(ll.shape[0], 1)))
    return res
