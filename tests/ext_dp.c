/* TEST INFRASTRUCTURE ONLY -- the scalar twin of the two DP routines of tests/ext_ref.py (bwa 0.7.17's ksw_extend2 and
   the score of ksw_align2), cell by cell as include/debwt_b200.h states them.  tests/ext_ref.py compiles it with gcc into
   a temporary directory and checks it against its Python loops; the regions reference calls it for speed.
   q: query codes 0..4, t: target codes 0..3. */
#include <stdint.h>
#include <stdlib.h>

static unsigned long long n_cells;   /* DP cells computed since the library was loaded */

unsigned long long ext_cells(void) { return n_cells; }

static int sc(int a, int b, uint8_t t, uint8_t q) { return q > 3 ? -1 : t == q ? a : -b; }

/* out: qle, tle, gtle, gscore, max_off; returns max (h0 > 0) */
int ext_extend(int qlen, const uint8_t* q, int tlen, const uint8_t* t, int a, int b, int o_del, int e_del, int o_ins, int e_ins, int w,
               int end_bonus, int zdrop, int h0, int* out) {
    const int oe_del = o_del + e_del, oe_ins = o_ins + e_ins;
    int* H = calloc((size_t)qlen + 2, sizeof(int));
    int* E = calloc((size_t)qlen + 2, sizeof(int));
    H[0] = h0;
    if (qlen >= 1) H[1] = h0 > oe_ins ? h0 - oe_ins : 0;
    for (int j = 2; j <= qlen && H[j - 1] > e_ins; ++j) H[j] = H[j - 1] - e_ins;
    int max_ins = (int)((double)(qlen * a + end_bonus - o_ins) / e_ins + 1.);
    max_ins = max_ins > 1 ? max_ins : 1;
    w = w < max_ins ? w : max_ins;
    int max_del = (int)((double)(qlen * a + end_bonus - o_del) / e_del + 1.);
    max_del = max_del > 1 ? max_del : 1;
    w = w < max_del ? w : max_del;
    int max = h0, max_i = -1, max_j = -1, max_ie = -1, gscore = -1, max_off = 0, beg = 0, end = qlen;
    for (int i = 0; i < tlen; ++i) {
        int f = 0, h1, m = 0, mj = -1, j;
        if (beg < i - w) beg = i - w;
        if (end > i + w + 1) end = i + w + 1;
        if (end > qlen) end = qlen;
        if (beg == 0) {
            long long v = (long long)h0 - (o_del + (long long)e_del * (i + 1));
            h1 = v > 0 ? (int)v : 0;
        } else h1 = 0;
        n_cells += end > beg ? (unsigned long long)(end - beg) : 0;
        for (j = beg; j < end; ++j) {
            int M = H[j], e = E[j], h, x;
            H[j] = h1;
            M = M ? M + sc(a, b, t[i], q[j]) : 0;
            h = M > e ? M : e;
            h = h > f ? h : f;
            h1 = h;
            mj = m > h ? mj : j;
            m = m > h ? m : h;
            x = M - oe_del; x = x > 0 ? x : 0;
            e -= e_del; e = e > x ? e : x;
            E[j] = e;
            x = M - oe_ins; x = x > 0 ? x : 0;
            f -= e_ins; f = f > x ? f : x;
        }
        H[end] = h1; E[end] = 0;
        if (j == qlen) {
            max_ie = gscore > h1 ? max_ie : i;
            gscore = gscore > h1 ? gscore : h1;
        }
        if (m == 0) break;
        if (m > max) {
            max = m, max_i = i, max_j = mj;
            max_off = max_off > abs(mj - i) ? max_off : abs(mj - i);
        } else if (zdrop > 0) {
            long long di = i - max_i, dj = mj - max_j;
            if (di > dj) {
                if (max - m - (di - dj) * e_del > zdrop) break;
            } else if (max - m - (dj - di) * e_ins > zdrop) break;
        }
        for (j = beg; j < end && H[j] == 0 && E[j] == 0; ++j) {}
        beg = j;
        for (j = end; j >= beg && H[j] == 0 && E[j] == 0; --j) {}
        end = j + 2 < qlen ? j + 2 : qlen;
    }
    free(H); free(E);
    out[0] = max_j + 1; out[1] = max_i + 1; out[2] = max_ie + 1; out[3] = gscore; out[4] = max_off;
    return max;
}

/* Gotoh local alignment score: H >= 0, gaps open from H, E over the target (deletion), F over the query (insertion) */
int ext_seed_sw(int qlen, const uint8_t* q, int tlen, const uint8_t* t, int a, int b, int o_del, int e_del, int o_ins, int e_ins) {
    int* H = calloc((size_t)qlen + 1, sizeof(int));     /* H[j + 1] = H(i - 1, j) */
    int* E = calloc((size_t)qlen + 1, sizeof(int));     /* E[j] = E(i, j) */
    int best = 0;
    n_cells += (unsigned long long)qlen * (unsigned long long)tlen;
    for (int i = 0; i < tlen; ++i) {
        int diag = 0, left = 0, f = 0;                  /* diag = H(i - 1, j - 1), left = H(i, j - 1), f = F(i, j) */
        for (int j = 0; j < qlen; ++j) {
            int up = H[j + 1], h = diag + sc(a, b, t[i], q[j]), x;
            x = left - (o_ins + e_ins); f -= e_ins; f = f > x ? f : x; f = f > 0 ? f : 0;
            if (j == 0) f = 0;
            h = h > E[j] ? h : E[j];
            h = h > f ? h : f;
            h = h > 0 ? h : 0;
            best = best > h ? best : h;
            x = h - (o_del + e_del); E[j] -= e_del; E[j] = E[j] > x ? E[j] : x; E[j] = E[j] > 0 ? E[j] : 0;
            diag = up;
            left = h;
            H[j + 1] = h;
        }
    }
    free(H); free(E);
    return best;
}
