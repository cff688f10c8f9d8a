/* greedy_nl.c -- CPU oracles of the greedy-edge constructor; see greedy_nl.h. */
#include "greedy_nl.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

typedef struct {
    float d;
    int32_t lo, hi;
} gkey;

static int key_less(gkey a, gkey b)
{
    return a.d < b.d || (a.d == b.d && (a.lo < b.lo || (a.lo == b.lo && a.hi < b.hi)));
}

static float gdist(const float *x, const float *y, int nint, int32_t a, int32_t b)
{
    return nint ? (float)tlo_dist_nint(x[a], y[a], x[b], y[b]) : tlo_dist_f32(x[a], y[a], x[b], y[b]);
}

static gkey mkkey(float d, int32_t a, int32_t b)
{
    gkey k = {d, a < b ? a : b, a < b ? b : a};
    return k;
}

/* adj: 2 slots per city, the closing edge included */
static void emit(int32_t n, const int32_t *adj, int32_t *out)
{
    if (n <= 3) {
        for (int32_t k = 0; k < n; ++k) out[k] = k;
        return;
    }
    int32_t prev = 0, cur = adj[0] < adj[1] ? adj[0] : adj[1];
    out[0] = 0;
    for (int32_t k = 1; k < n; ++k) {
        out[k] = cur;
        const int32_t nx = adj[2 * cur] == prev ? adj[2 * cur + 1] : adj[2 * cur];
        prev = cur;
        cur = nx;
    }
}

/* ---- (a) brute force ------------------------------------------------------------------------------------ */

typedef struct {
    gkey k;
} gedge;

static int cmp_edge(const void *pa, const void *pb)
{
    const gkey a = ((const gedge *)pa)->k, b = ((const gedge *)pb)->k;
    return key_less(a, b) ? -1 : (key_less(b, a) ? 1 : 0);
}

static int32_t uf_find(int32_t *par, int32_t a)
{
    while (par[a] != a) {
        par[a] = par[par[a]];
        a = par[a];
    }
    return a;
}

void tlo_greedy_brute(int32_t n, const float *x, const float *y, int nint, int32_t *out)
{
    if (n <= 3) {
        emit(n, NULL, out);
        return;
    }
    const int64_t m = (int64_t)n * (n - 1) / 2;
    gedge *e = malloc(sizeof(gedge) * m);
    int32_t *par = malloc(sizeof(int32_t) * n), *deg = calloc(n, sizeof(int32_t)), *adj = malloc(sizeof(int32_t) * 2 * n);
    int64_t c = 0;
    for (int32_t b = 1; b < n; ++b)
        for (int32_t a = 0; a < b; ++a) e[c++].k = mkkey(gdist(x, y, nint, a, b), a, b);
    qsort(e, m, sizeof(gedge), cmp_edge);
    for (int32_t v = 0; v < n; ++v) par[v] = v;
    int32_t taken = 0;
    for (int64_t t = 0; t < m && taken < n - 1; ++t) {
        const int32_t a = e[t].k.lo, b = e[t].k.hi;
        if (deg[a] >= 2 || deg[b] >= 2) continue;
        const int32_t ra = uf_find(par, a), rb = uf_find(par, b);
        if (ra == rb) continue;
        par[ra] = rb;
        adj[2 * a + deg[a]++] = b;
        adj[2 * b + deg[b]++] = a;
        ++taken;
    }
    int32_t ends[2], ne = 0;
    for (int32_t v = 0; v < n; ++v)
        if (deg[v] < 2) ends[ne++] = v;
    adj[2 * ends[0] + 1] = ends[1];
    adj[2 * ends[1] + 1] = ends[0];
    emit(n, adj, out);
    free(e);
    free(par);
    free(deg);
    free(adj);
}

/* ---- (b) Bentley's lazy greedy on a uniform grid ------------------------------------------------------------ */

typedef struct {
    int32_t n, nint;
    const float *x, *y;
    double x0, y0, cs; /* grid origin and cell size */
    double slack;      /* bound on the f64 rounding of a cell border */
    int32_t gx, gy;
    int32_t *start, *cnt, *cells, *cell_of, *slot;
    int32_t *deg, *other;
} lazy_t;

static int32_t clampi(int32_t v, int32_t lo, int32_t hi) { return v < lo ? lo : (v > hi ? hi : v); }

static void grid_remove(lazy_t *L, int32_t u)
{
    const int32_t c = L->cell_of[u], s = L->slot[u];
    const int32_t last = L->cells[L->start[c] + L->cnt[c] - 1];
    L->cells[L->start[c] + s] = last;
    L->slot[last] = s;
    L->cnt[c]--;
}

/* nearest eligible city of free city u in key order; returns -1 when there is none */
static int32_t nearest_eligible(const lazy_t *L, int32_t u, float *dout)
{
    const double px = L->x[u], py = L->y[u];
    const int32_t cx = clampi((int32_t)((px - L->x0) / L->cs), 0, L->gx - 1);
    const int32_t cy = clampi((int32_t)((py - L->y0) / L->cs), 0, L->gy - 1);
    int32_t best = -1;
    float bd = 0.0f;
    for (int32_t r = 0;; ++r) {
        for (int32_t iy = cy - r; iy <= cy + r; ++iy) {
            if (iy < 0 || iy >= L->gy) continue;
            const int32_t step = (iy == cy - r || iy == cy + r) ? 1 : 2 * r;
            for (int32_t ix = cx - r; ix <= cx + r; ix += step) {
                if (ix < 0 || ix >= L->gx) continue;
                const int32_t c = iy * L->gx + ix;
                for (int32_t t = 0; t < L->cnt[c]; ++t) {
                    const int32_t w = L->cells[L->start[c] + t];
                    if (w == u || w == L->other[u]) continue;
                    const float d = gdist(L->x, L->y, L->nint, u, w);
                    if (best < 0 || d < bd || (d == bd && w < best)) {
                        best = w;
                        bd = d;
                    }
                }
            }
        }
        const int done_x = cx - r <= 0 && cx + r >= L->gx - 1, done_y = cy - r <= 0 && cy + r >= L->gy - 1;
        if (done_x && done_y) break;
        /* every unsearched city lies outside the square of cells cx-r..cx+r x cy-r..cy+r */
        double gap = INFINITY;
        if (cx - r > 0) gap = fmin(gap, px - (L->x0 + (cx - r) * L->cs));
        if (cx + r < L->gx - 1) gap = fmin(gap, L->x0 + (cx + r + 1) * L->cs - px);
        if (cy - r > 0) gap = fmin(gap, py - (L->y0 + (cy - r) * L->cs));
        if (cy + r < L->gy - 1) gap = fmin(gap, L->y0 + (cy + r + 1) * L->cs - py);
        gap -= L->slack; /* cell indices and borders are rounded in f64 */
        const double lower = L->nint ? gap - 0.5 - 1e-9 * gap : gap * (1.0 - ldexp(1.0, -20));
        if (best >= 0 && (double)bd < lower) break;
    }
    *dout = bd;
    return best;
}

typedef struct {
    gkey k;
    int32_t u, v; /* entry of free city u: its nearest eligible city v when pushed */
} hentry;

static void heap_push(hentry *h, int64_t *hn, hentry e)
{
    int64_t i = (*hn)++;
    while (i > 0) {
        const int64_t p = (i - 1) / 2;
        if (!key_less(e.k, h[p].k)) break;
        h[i] = h[p];
        i = p;
    }
    h[i] = e;
}

static hentry heap_pop(hentry *h, int64_t *hn)
{
    const hentry top = h[0], e = h[--(*hn)];
    int64_t i = 0;
    for (;;) {
        int64_t c = 2 * i + 1;
        if (c >= *hn) break;
        if (c + 1 < *hn && key_less(h[c + 1].k, h[c].k)) ++c;
        if (!key_less(h[c].k, e.k)) break;
        h[i] = h[c];
        i = c;
    }
    if (*hn > 0) h[i] = e;
    return top;
}

static void push_nearest(const lazy_t *L, hentry *h, int64_t *hn, int32_t u)
{
    float d;
    const int32_t v = nearest_eligible(L, u, &d);
    if (v < 0) return;
    hentry e = {mkkey(d, u, v), u, v};
    heap_push(h, hn, e);
}

void tlo_greedy_lazy(int32_t n, const float *x, const float *y, int nint, int32_t *out)
{
    if (n <= 3) {
        emit(n, NULL, out);
        return;
    }
    lazy_t L;
    memset(&L, 0, sizeof L);
    L.n = n;
    L.nint = nint;
    L.x = x;
    L.y = y;
    double x1 = x[0], y1 = y[0];
    L.x0 = x[0];
    L.y0 = y[0];
    for (int32_t i = 1; i < n; ++i) {
        L.x0 = fmin(L.x0, x[i]);
        x1 = fmax(x1, x[i]);
        L.y0 = fmin(L.y0, y[i]);
        y1 = fmax(y1, y[i]);
    }
    /* about two cities per cell */
    const double w = fmax(x1 - L.x0, 0.0), hgt = fmax(y1 - L.y0, 0.0);
    double cs = sqrt(2.0 * fmax(w * hgt, 1e-300) / n);
    if (!(cs > 0.0) || w / cs > 4.0 * n || hgt / cs > 4.0 * n) cs = fmax(w, hgt) / n;
    if (!(cs > 0.0)) cs = 1.0;
    L.cs = cs;
    L.slack = 1e-13 * (fabs(L.x0) + fabs(L.y0) + w + hgt + cs);
    L.gx = (int32_t)fmin(w / cs, 4.0 * n) + 1;
    L.gy = (int32_t)fmin(hgt / cs, 4.0 * n) + 1;
    const int64_t ncell = (int64_t)L.gx * L.gy;
    L.start = calloc(ncell + 1, sizeof(int32_t));
    L.cnt = calloc(ncell, sizeof(int32_t));
    L.cells = malloc(sizeof(int32_t) * n);
    L.cell_of = malloc(sizeof(int32_t) * n);
    L.slot = malloc(sizeof(int32_t) * n);
    L.deg = calloc(n, sizeof(int32_t));
    L.other = malloc(sizeof(int32_t) * n);
    for (int32_t u = 0; u < n; ++u) {
        const int32_t cx = clampi((int32_t)((x[u] - L.x0) / cs), 0, L.gx - 1);
        const int32_t cy = clampi((int32_t)((y[u] - L.y0) / cs), 0, L.gy - 1);
        L.cell_of[u] = cy * L.gx + cx;
        L.cnt[L.cell_of[u]]++;
        L.other[u] = u;
    }
    for (int64_t c = 0; c < ncell; ++c) L.start[c + 1] = L.start[c] + L.cnt[c];
    memset(L.cnt, 0, sizeof(int32_t) * ncell);
    for (int32_t u = 0; u < n; ++u) {
        const int32_t c = L.cell_of[u];
        L.slot[u] = L.cnt[c]++;
        L.cells[L.start[c] + L.slot[u]] = u;
    }
    int32_t *adj = malloc(sizeof(int32_t) * 2 * n);
    hentry *h = malloc(sizeof(hentry) * ((int64_t)n + 8));
    int64_t hn = 0;
    for (int32_t u = 0; u < n; ++u) push_nearest(&L, h, &hn, u);
    int32_t taken = 0;
    while (taken < n - 1 && hn > 0) {
        const hentry e = heap_pop(h, &hn);
        const int32_t u = e.u, v = e.v;
        if (L.deg[u] >= 2) continue; /* u left the free set: its entry goes */
        if (L.deg[v] >= 2 || v == L.other[u]) { /* stale: search again */
            push_nearest(&L, h, &hn, u);
            continue;
        }
        const int32_t a = L.other[u], b = L.other[v];
        adj[2 * u + L.deg[u]++] = v;
        adj[2 * v + L.deg[v]++] = u;
        L.other[a] = b;
        L.other[b] = a;
        ++taken;
        if (L.deg[u] == 2) grid_remove(&L, u);
        if (L.deg[v] == 2) grid_remove(&L, v);
        if (L.deg[u] < 2) push_nearest(&L, h, &hn, u); /* v keeps its own entry, checked when popped */
    }
    int32_t ends[2], ne = 0;
    for (int32_t v = 0; v < n && ne < 2; ++v)
        if (L.deg[v] < 2) ends[ne++] = v;
    adj[2 * ends[0] + 1] = ends[1];
    adj[2 * ends[1] + 1] = ends[0];
    emit(n, adj, out);
    free(L.start);
    free(L.cnt);
    free(L.cells);
    free(L.cell_of);
    free(L.slot);
    free(L.deg);
    free(L.other);
    free(adj);
    free(h);
}
