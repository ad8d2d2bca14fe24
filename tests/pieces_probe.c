/* TEST INFRASTRUCTURE ONLY: the oracle's own token loop and N re-insertion (orc_reconstruct in oracle/sccg_oracle.c,
 * decompression.cpp:210-252), reporting what they do instead of the bytes they produce, for the reference implementation of
 * sccg_archive_variants in tests/variants_lib.py.  The oracle source is included as it is, so the token forms it accepts
 * (stoi, a '(' inside the target) decode exactly as there.
 *   pieces: (x, p, l) per token that copies l >= 1 bytes: record-stream position x, position p in the prepared reference
 *   ins:    the positions of D at which the N re-insertion put an N, ascending
 * Returns the rc of orc_reconstruct for the same input (0: it decodes). */
#include "../oracle/sccg_oracle.c"

int orc_reconstruct_pieces(const char* ref, long nr, const char* enc, long ne, const char* n_idx, long nn,
                           long** pieces, long* n_pieces, long* rec_len, long** ins, long* n_ins) {
    ivec ns = {0, 0, 0};
    long np = 0, cap = 0, x = 0, ni = 0;
    long *pc = 0, *iv = 0;
    int rc = 0;
    if (parse_run_list(n_idx, nn, &ns)) { rc = 1; goto done; }
    {
        uint64_t i = 0; int prev_abs_start = 0;
        while (i < (uint64_t)ne) {
            if (enc[i] == '(') {
                uint64_t end_pos = ufind(enc, ne, ')', i);
                uint64_t comma_pos = ufind(enc, ne, ',', i);
                long b1, e1, b2, e2; int ok1, ok2;
                if (!substr_rng(ne, i + 1, comma_pos - i - 1, &b1, &e1)) { rc = 1; goto done; }
                int delta = orc_stoi(enc + b1, e1 - b1, &ok1);
                if (!ok1) { rc = 1; goto done; }
                if (!substr_rng(ne, comma_pos + 1, end_pos - comma_pos - 1, &b2, &e2)) { rc = 1; goto done; }
                int length = orc_stoi(enc + b2, e2 - b2, &ok2);
                if (!ok2) { rc = 1; goto done; }
                int absolute_start = prev_abs_start + delta;
                prev_abs_start = absolute_start;
                if (absolute_start + length > (int)nr) { rc = 3; goto done; }
                long cb, ce;
                if (!substr_rng(nr, (uint64_t)(int64_t)absolute_start, (uint64_t)(int64_t)length, &cb, &ce)) { rc = 1; goto done; }
                if (ce > cb) {
                    if (np + 3 > cap) { cap = cap ? 2 * cap : 3 * 1024; pc = (long*)realloc(pc, sizeof(long) * (size_t)cap); }
                    pc[np++] = x; pc[np++] = cb; pc[np++] = ce - cb;
                }
                x += ce - cb;
                if (end_pos == NPOS) { rc = 1; goto done; }
                i = end_pos + 1;
            } else {
                ++x; ++i;
            }
        }
    }
    {
        long temp_index = 0, n_pos = 0;
        int total = (int)(x + ns.n);
        iv = (long*)malloc(sizeof(long) * (size_t)(ns.n + 1));
        for (int i = 0; i < total; ++i) {
            if (n_pos < ns.n && ns.d[n_pos] == i) { iv[ni++] = i; ++n_pos; }
            else {
                if (temp_index > x) { rc = 4; goto done; }
                temp_index++;
            }
        }
    }
done:
    free(ns.d);
    if (rc != 0) { free(pc); free(iv); pc = 0; iv = 0; np = 0; ni = 0; }
    *pieces = pc; *n_pieces = np / 3; *rec_len = x; *ins = iv; *n_ins = ni;
    return rc;
}
