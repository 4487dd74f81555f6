/*
 * stats_oracle.c -- TEST INFRASTRUCTURE: the serial reference of the strand / quality pass (amplipy_b200/csrc/amp_ivar.cuh).
 * It adds oracle_pileup_stats_batch to the C oracle (oracle/amplipy_oracle.c, included unchanged): the literal pair-list walk of
 * pileup_read (AmpliPy.py:706-753) once more, recording for every event the count matrix receives its strand and quality.
 */
#include "../oracle/amplipy_oracle.c"

/* one read; returns 0 ok, F_ERROR where pileup_read stops (the events before that point count, as they do there) */
static int stats_read(int64_t* rev, int64_t* qsum, int L, int32_t ref_start, const cig_t* c, int nc, const char* query_seq,
                      const uint8_t* query_qual, int l_seq, int min_quality, int is_rev, int32_t* pq, int32_t* pr, int64_t* nev,
                      int64_t ev_cap, int32_t* ev_pos, int32_t* ev_rev, int32_t* ev_qual, int8_t* ev_head, int64_t* ev_off,
                      char* ev_chars, int64_t chars_cap) {
    int query_start = query_alignment_start(c, nc);
    int query_end = query_alignment_end(c, nc, l_seq);
    int ref_end = ref_start + ref_len_of(c, nc);
    int np = 0, q = 0, r = ref_start;
    for (int k = 0; k < nc; ++k) {
        int op = c[k].op, n = c[k].n;
        if (op == OP_M || op == OP_EQ || op == OP_X) { for (int j = 0; j < n; ++j) { pq[np] = q + j; pr[np] = r + j; np++; } q += n; r += n; }
        else if (op == OP_I || op == OP_S || op == OP_P) { for (int j = 0; j < n; ++j) { pq[np] = q + j; pr[np] = -1; np++; } q += n; }
        else if (op == OP_D || op == OP_N) { for (int j = 0; j < n; ++j) { pq[np] = -1; pr[np] = r + j; np++; } r += n; }
    }
    if (q > l_seq) return F_ERROR;
    if (r > L) return F_ERROR;
    int i = 0;
    while (i < np) {
        int q_pos = pq[i], r_pos = pr[i]; i++;
        if (q_pos < 0) { rev[5 * (int64_t)L + r_pos] += is_rev; }                 /* 714-715: no quality */
        else if (query_qual[q_pos] < min_quality) continue;
        else if (q_pos < query_start) continue;
        else if (q_pos >= query_end) break;
        else if (r_pos < 0) {
            int q0 = q_pos;
            while (r_pos < 0 && q_pos < query_end && query_qual[q_pos] >= min_quality) {
                if (i >= np) return F_ERROR;
                q_pos = pq[i]; r_pos = pr[i]; i++;
                if (q_pos < 0) break;
            }
            int s_begin, s_end, head = 0;
            if (r_pos == 0) {
                if (q_pos < 0) return F_ERROR;
                s_begin = q0; s_end = q_pos + 1; head = 1;                       /* 735-736 */
            } else {
                s_begin = q0 - 1; if (s_begin < 0) s_begin += l_seq;
                if (s_begin < 0) s_begin = 0;
                s_end = (q_pos < 0) ? l_seq : q_pos;
            }
            if (s_end > l_seq) s_end = l_seq;
            int slen = s_end - s_begin; if (slen < 0) slen = 0;
            int ref_insertion_pos;
            if (r_pos < 0) ref_insertion_pos = ref_end;
            else { ref_insertion_pos = r_pos; i -= 1; }
            ref_insertion_pos = ref_insertion_pos - 1 > 0 ? ref_insertion_pos - 1 : 0;
            if (ref_insertion_pos >= L) return F_ERROR;
            const int eq = query_qual[q0];                                        /* the event's quality */
            int one = (slen == 1) ? sym_channel(query_seq[s_begin]) : -1;
            if (one >= 0) { rev[one * (int64_t)L + ref_insertion_pos] += is_rev; qsum[one * (int64_t)L + ref_insertion_pos] += eq; }
            else {
                int64_t e = (*nev)++;
                if (e < ev_cap) {
                    ev_pos[e] = ref_insertion_pos; ev_rev[e] = is_rev; ev_qual[e] = eq; ev_head[e] = (int8_t)head;
                    if (ev_off[e] + slen <= chars_cap) memcpy(ev_chars + ev_off[e], query_seq + s_begin, (size_t)slen);
                    ev_off[e + 1] = ev_off[e] + slen;
                }
            }
        } else if (query_qual[q_pos] >= min_quality) {
            int ch = sym_channel(query_seq[q_pos]);
            if (ch < 0) return F_ERROR;
            rev[ch * (int64_t)L + r_pos] += is_rev; qsum[ch * (int64_t)L + r_pos] += query_qual[q_pos];
        }
    }
    return 0;
}

/*
 * rev / qsum: int64 [6][L] (zeroed by the caller).  Insertion events in read order: ev_pos, ev_rev (0/1), ev_qual, ev_head
 * (1: the key of 735-736), key e = ev_chars[ev_off[e], ev_off[e + 1]); ev_off[0] = 0 on entry.  Row layout and skipping as in
 * oracle_pileup_batch.  Returns the number of events; if it is larger than ev_cap, or ev_off[min(n, ev_cap)] > chars_cap, call
 * again with more room.
 */
int64_t oracle_pileup_stats_batch(int64_t N, const int32_t* pos, const uint16_t* flag, const uint32_t* cig_off, const uint32_t* cigar,
                                  const int32_t* ncig, int row_stride3, const uint8_t* skip_flags, const uint32_t* seq_off,
                                  const uint8_t* seq, const uint32_t* qual_off, const uint8_t* qual, int L, int min_quality,
                                  int64_t* rev, int64_t* qsum, int64_t ev_cap, int32_t* ev_pos, int32_t* ev_rev, int32_t* ev_qual,
                                  int8_t* ev_head, int64_t* ev_off, char* ev_chars, int64_t chars_cap) {
    int64_t nev = 0;
    cig_t* c = NULL; int ccap = 0; char* s = NULL; int32_t* pq = NULL; int32_t* pr = NULL; int scap = 0, pcap = 0;
    for (int64_t i = 0; i < N; ++i) {
        if (skip_flags && (skip_flags[i] & (F_SKIPPED | F_ERROR))) continue;
        const uint32_t* row; int nc;
        if (row_stride3) { row = cigar + (size_t)cig_off[i] + 3 * (size_t)i; nc = ncig[i]; }
        else { row = cigar + cig_off[i]; nc = (int)(cig_off[i + 1] - cig_off[i]); }
        if ((flag[i] & 4) || nc == 0) continue;
        int l_seq = (int)(qual_off[i + 1] - qual_off[i]);
        if (nc > ccap) { ccap = 2 * nc; c = (cig_t*)realloc(c, sizeof(cig_t) * ccap); }
        int npairs = 0;
        for (int k = 0; k < nc; ++k) { c[k].op = (int)(row[k] & 15); c[k].n = (int)(row[k] >> 4); if (c[k].op != OP_H) npairs += c[k].n; }
        if (l_seq + 1 > scap) { scap = 2 * (l_seq + 1); s = (char*)realloc(s, scap); }
        if (npairs + 1 > pcap) { pcap = 2 * (npairs + 1); pq = (int32_t*)realloc(pq, sizeof(int32_t) * pcap); pr = (int32_t*)realloc(pr, sizeof(int32_t) * pcap); }
        const uint8_t* sp = seq + seq_off[i];
        for (int j = 0; j < l_seq; ++j) s[j] = NIB2CHAR[(sp[j >> 1] >> ((~j & 1) << 2)) & 15];
        stats_read(rev, qsum, L, pos[i], c, nc, s, qual + qual_off[i], l_seq, min_quality, (flag[i] & 16) ? 1 : 0, pq, pr, &nev, ev_cap,
                   ev_pos, ev_rev, ev_qual, ev_head, ev_off, ev_chars, chars_cap);
    }
    free(c); free(s); free(pq); free(pr);
    return nev;
}
