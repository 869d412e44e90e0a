/* cluster_ref.c -- CPU reference of itsx_cluster (DESIGN.md §6), written from the definition alone.
 *
 * Brute force: every class, in processing order, is compared with every earlier centroid whose length is within D of
 * its own; there is no seed filter, so it checks both the greedy and the losslessness of the GPU's candidate
 * generation.  The only thing shared with the library is the acceptance table D(L) (itsx_cluster_dtable).
 * Edit distance: unit-cost Levenshtein over normalised residues (upper case, U = T, IUPAC symbols are ordinary letters,
 * complement of the reverse strand as the derep takes it), over the cells within d of the diagonal only (a path through
 * any other costs more than d), stopped once a whole row exceeds d. */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

static unsigned char norm(unsigned char c)
{
    if (c >= 'a' && c <= 'z') c -= 32;
    return c == 'U' ? 'T' : c;
}
static unsigned char comp(unsigned char c)
{
    static const char *from = "ACGTRYMKHDBV", *to = "TGCAYRKMDHVB";
    const char *p = strchr(from, c);
    return p && c ? (unsigned char)to[p - from] : c;
}

/* ed(a, b) if <= d, else d + 1 */
static int ed_within(const unsigned char *a, int n, const unsigned char *b, int m, int d, int *prev, int *cur)
{
    const int INF = d + 1;
    if (abs(n - m) > d) return INF;
    for (int j = 0; j <= m; j++) prev[j] = j <= d ? j : INF;
    for (int i = 1; i <= n; i++) {
        int rowmin = INF;
        const int j0 = i - d > 0 ? i - d : 0, j1 = i + d < m ? i + d : m;
        for (int j = j0; j <= j1; j++) {
            int x = j <= i - 1 + d ? prev[j] + 1 : INF;                  /* (i-1, j), outside the band beyond i-1+d */
            if (j > 0) {
                const int diag = prev[j - 1] + (a[i - 1] != b[j - 1]);
                if (diag < x) x = diag;
                if (j - 1 >= j0 && cur[j - 1] + 1 < x) x = cur[j - 1] + 1;
            }
            if (x > INF) x = INF;
            cur[j] = x;
            if (x < rowmin) rowmin = x;
        }
        if (rowmin > d) return INF;
        int *t = prev; prev = cur; cur = t;
    }
    return prev[m];
}

/* seq/off: the reads; first[u]: first read of unique u; order[r]: unique processed r-th; D[0..lmax].
 * Out per unique: crow (centroid row), strand (0 '+', 1 '-'), ed; uor[row] = unique of the row's centroid.
 * Returns the number of centroids. */
int64_t ref_cluster(const uint8_t *seq, const int64_t *off, const int32_t *first, int64_t nu, const int32_t *order,
                    const int32_t *D, int32_t lmax, int32_t *crow, uint8_t *strand, int32_t *ed, int32_t *uor)
{
    unsigned char **fw = malloc(sizeof(*fw) * (nu ? nu : 1)), **rv = malloc(sizeof(*rv) * (nu ? nu : 1));
    int *len = malloc(sizeof(int) * (nu ? nu : 1));
    int64_t *cent = malloc(sizeof(int64_t) * (nu ? nu : 1));      /* unique of every centroid, in row order */
    int *prev = malloc(sizeof(int) * (lmax + 2)), *cur = malloc(sizeof(int) * (lmax + 2));
    for (int64_t u = 0; u < nu; u++) {
        const uint8_t *s = seq + off[first[u]];
        const int L = (int)(off[first[u] + 1] - off[first[u]]);
        len[u] = L;
        fw[u] = malloc(L + 1);
        rv[u] = malloc(L + 1);
        for (int m = 0; m < L; m++) {
            fw[u][m] = norm(s[m]);
            rv[u][L - 1 - m] = comp(norm(s[m]));
        }
    }
    int64_t nc = 0;
    for (int64_t r = 0; r < nu; r++) {
        const int64_t u = order[r];
        int64_t best = -1;
        long long bn = 0, bd = 1;
        int bed = 0, bst = 0;
        for (int64_t k = 0; k < nc; k++) {
            const int64_t v = cent[k];
            const int L = len[u] > len[v] ? len[u] : len[v], d = D[L];
            if (abs(len[u] - len[v]) > d) continue;
            const int ep = ed_within(fw[u], len[u], fw[v], len[v], d, prev, cur);
            const int em = ed_within(rv[u], len[u], fw[v], len[v], d, prev, cur);
            const int e = ep <= em ? ep : em;
            if (e > d) continue;
            if (best < 0 || (long long)(L - e) * bd > bn * L) { best = k; bn = L - e; bd = L; bed = e; bst = em < ep; }
        }
        if (best < 0) {
            crow[u] = (int32_t)nc;
            strand[u] = 0;
            ed[u] = 0;
            uor[nc] = (int32_t)u;
            cent[nc++] = u;
        } else {
            crow[u] = (int32_t)best;
            strand[u] = (uint8_t)bst;
            ed[u] = bed;
        }
    }
    for (int64_t u = 0; u < nu; u++) { free(fw[u]); free(rv[u]); }
    free(fw); free(rv); free(len); free(cent); free(prev); free(cur);
    return nc;
}

/* the number of unordered pairs of distinct uniques of the same group (group[u]: sample or family of unique u) that are
 * accepted: min(ed(s_u, s_v), ed(rc(s_u), s_v)) <= D(max(len_u, len_v)).  Brute force over every pair of a group whose
 * lengths are within D; acceptance is symmetric, so this is the number of accepted edges whatever the order.  Only the
 * pairs whose first member is at a position in [a0, a1) of the (group, unique) order are counted, so that callers can
 * split the work. */
static int cmp_group(const void *x, const void *y)
{
    const int64_t *a = x, *b = y;       /* (group, unique) */
    return a[0] != b[0] ? (a[0] < b[0] ? -1 : 1) : (a[1] < b[1] ? -1 : a[1] > b[1]);
}
int64_t ref_accepted_pairs(const uint8_t *seq, const int64_t *off, const int32_t *first, int64_t nu, const int32_t *group,
                           const int32_t *D, int32_t lmax, int64_t a0, int64_t a1)
{
    int64_t *ix = malloc(sizeof(int64_t) * 2 * (nu ? nu : 1));
    unsigned char **fw = malloc(sizeof(*fw) * (nu ? nu : 1)), **rv = malloc(sizeof(*rv) * (nu ? nu : 1));
    int *len = malloc(sizeof(int) * (nu ? nu : 1));
    int *prev = malloc(sizeof(int) * (lmax + 2)), *cur = malloc(sizeof(int) * (lmax + 2));
    for (int64_t u = 0; u < nu; u++) {
        const uint8_t *s = seq + off[first[u]];
        const int L = (int)(off[first[u] + 1] - off[first[u]]);
        len[u] = L;
        fw[u] = malloc(L + 1);
        rv[u] = malloc(L + 1);
        for (int m = 0; m < L; m++) {
            fw[u][m] = norm(s[m]);
            rv[u][L - 1 - m] = comp(norm(s[m]));
        }
        ix[2 * u] = group[u];
        ix[2 * u + 1] = u;
    }
    qsort(ix, nu, 2 * sizeof(int64_t), cmp_group);
    int64_t n = 0;
    for (int64_t a = a0; a < a1 && a < nu; a++) {
        const int64_t u = ix[2 * a + 1];
        for (int64_t b = a + 1; b < nu && ix[2 * b] == ix[2 * a]; b++) {
            const int64_t v = ix[2 * b + 1];
            const int L = len[u] > len[v] ? len[u] : len[v], d = D[L];
            if (abs(len[u] - len[v]) > d) continue;
            if (ed_within(fw[u], len[u], fw[v], len[v], d, prev, cur) <= d ||
                ed_within(rv[u], len[u], fw[v], len[v], d, prev, cur) <= d)
                n++;
        }
    }
    for (int64_t u = 0; u < nu; u++) { free(fw[u]); free(rv[u]); }
    free(ix); free(fw); free(rv); free(len); free(prev); free(cur);
    return n;
}

/* the ed (<= d, else d + 1) of a, or of its reverse complement (rc = 1), against b, for tests of the greedy's inputs */
int ref_ed(const uint8_t *a, int n, const uint8_t *b, int m, int d, int rc)
{
    unsigned char *x = malloc(n + 1), *y = malloc(m + 1);
    int *prev = malloc(sizeof(int) * (m + 2)), *cur = malloc(sizeof(int) * (m + 2));
    for (int i = 0; i < n; i++) {
        if (rc) x[n - 1 - i] = comp(norm(a[i]));
        else x[i] = norm(a[i]);
    }
    for (int j = 0; j < m; j++) y[j] = norm(b[j]);
    int e = ed_within(x, n, y, m, d, prev, cur);
    free(x); free(y); free(prev); free(cur);
    return e;
}
