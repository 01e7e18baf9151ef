/*
 * Betti matching by union-find -- TEST INFRASTRUCTURE ONLY (tests/betti_oracle.py builds and loads it; the product
 * package never does).
 *
 * A sequential restatement of dilabhelmholtzoct_b200/csrc/betti_kernel.cuh: elder-rule Kruskal passes for the
 * barcodes and the image barcodes, then the induced matching and its cost.  It reuses the cell values, keys and
 * pixel rules of oracle/topo_oracle.c (included, not modified) and is pinned against betti_matching_literal in
 * tests/betti_oracle.py (image persistence by a literal boundary-matrix reduction).
 */
#include "../oracle/topo_oracle.c"

/* value / top pixel of the edge at bitmap position pos */
static inline float edge_val_at(const float* f, int H, int W, uint32_t pos) {
    const int GW = 2 * W + 1, Y = (int)(pos / GW), X = (int)(pos % GW);
    return (Y & 1) ? vedge_val(f, W, (Y - 1) / 2, X / 2) : hedge_val(f, H, W, Y / 2, (X - 1) / 2);
}
static inline int32_t edge_top_at(const float* f, int H, int W, uint32_t pos) {
    const int GW = 2 * W + 1, Y = (int)(pos / GW), X = (int)(pos % GW);
    return (Y & 1) ? vedge_top(f, W, (Y - 1) / 2, X / 2) : hedge_top(f, H, W, Y / 2, (X - 1) / 2);
}

/*
 * Elder-rule Kruskal on the pixel graph with node keys from `nm` and edge keys from `em` (maps of one shape):
 * dim 0: vertices, edges ascending; dim 1: squares + OUTSIDE (id H*W, eldest), edges descending.  death[y] = bitmap
 * position of the edge at which node y dies, -1 for the root.  With nm = domain, em = codomain (dim 0) or
 * nm = codomain, em = domain (dim 1) the pairs are those of the image H_d(domain_t) -> H_d(codomain_t);
 * with nm == em they are the barcode.
 */
static void image_kruskal(const float* nm, const float* em, int H, int W, int dim, int32_t* death) {
    const int GW = 2 * W + 1, VW = W + 1, OUT = H * W;
    const int NN = dim == 0 ? (H + 1) * (W + 1) : H * W + 1;
    const int64_t nE = (int64_t)H * (W + 1) + (int64_t)(H + 1) * W;
    edge_t* E = (edge_t*)malloc(sizeof(edge_t) * (size_t)nE);
    int32_t* par = (int32_t*)malloc(sizeof(int32_t) * (size_t)NN);
    uint64_t* nkey = (uint64_t*)malloc(sizeof(uint64_t) * (size_t)NN);  /* smaller = elder */
    int ne = 0;
    for (int i = 0; i < H; ++i)
        for (int j = 0; j <= W; ++j) {
            E[ne].key = ((uint64_t)mono32(vedge_val(em, W, i, j)) << 32) | (uint32_t)(2 * j + (2 * i + 1) * GW);
            if (dim == 0) { E[ne].a = i * VW + j; E[ne].b = (i + 1) * VW + j; }
            else { E[ne].a = j == 0 ? OUT : i * W + j - 1; E[ne].b = j == W ? OUT : i * W + j; }
            ++ne;
        }
    for (int i = 0; i <= H; ++i)
        for (int j = 0; j < W; ++j) {
            E[ne].key = ((uint64_t)mono32(hedge_val(em, H, W, i, j)) << 32) | (uint32_t)(2 * j + 1 + (2 * i) * GW);
            if (dim == 0) { E[ne].a = i * VW + j; E[ne].b = i * VW + j + 1; }
            else { E[ne].a = i == 0 ? OUT : (i - 1) * W + j; E[ne].b = i == H ? OUT : i * W + j; }
            ++ne;
        }
    qsort(E, (size_t)ne, sizeof(edge_t), cmp_edge_asc);
    for (int k = 0; k < NN; ++k) {
        par[k] = k; death[k] = -1;
        if (dim == 0) nkey[k] = ((uint64_t)mono32(vertex_val_top(nm, H, W, k / VW, k % VW, NULL)) << 32) | (uint32_t)(2 * (k % VW) + 2 * (k / VW) * GW);
        else nkey[k] = k == OUT ? 0ull : ~(((uint64_t)mono32(nm[k]) << 32) | (uint32_t)k);
    }
    for (int s = 0; s < ne; ++s) {
        const edge_t* e = &E[dim == 0 ? s : ne - 1 - s];
        int32_t ra = uf_find(par, e->a), rb = uf_find(par, e->b);
        if (ra == rb) continue;
        int32_t dead = nkey[ra] > nkey[rb] ? ra : rb, live = dead == ra ? rb : ra;
        par[dead] = live;
        death[dead] = (int32_t)(uint32_t)e->key;
    }
    free(E); free(par); free(nkey);
}

/* keep death[y] only where the interval [birth, death) it stands for is non-empty (strictly positive persistence) */
static void keep_positive(const float* nm, const float* em, int H, int W, int dim, int32_t* death) {
    const int VW = W + 1, NN = dim == 0 ? (H + 1) * (W + 1) : H * W + 1;
    for (int y = 0; y < NN; ++y) {
        if (death[y] < 0) continue;
        const float ev = edge_val_at(em, H, W, (uint32_t)death[y]);
        const int keep = dim == 0 ? mono32(vertex_val_top(nm, H, W, y / VW, y % VW, NULL)) < mono32(ev)
                                  : mono32(ev) < mono32(nm[y]);
        if (!keep) death[y] = -1;
    }
}

/* (creator, destroyer) pixels of the barcode interval stored at node y of map f */
static void interval_pixels(const float* f, int H, int W, int dim, int y, int32_t pos, int32_t* cre, int32_t* des) {
    const int VW = W + 1;
    if (dim == 0) { vertex_val_top(f, H, W, y / VW, y % VW, cre); *des = edge_top_at(f, H, W, (uint32_t)pos); }
    else { *cre = edge_top_at(f, H, W, (uint32_t)pos); *des = y; }
}

/*
 * Betti matching of one prediction map L and one target map G (Stucki et al., ICML 2023) in dimension dim, by four
 * Kruskal passes: the barcodes L -> L and G -> G and the images L -> C and G -> C, C = min(L, G).  An L interval
 * and a G interval are matched when their image intervals (linked to them by the birth cell) die at the same cell
 * of C; the essential H0 classes are always matched.  Records in the order of the node that owns the interval
 * (dim 0: birth vertex, dim 1: death square), the essential H0 pair last among the matched ones.
 * matched[cap][4], up[cap][2], ut[cap][2]; counts[3] = (matched, unmatched pred, unmatched target); *cost =
 * sum matched (bL - bG)^2 + (dL - dG)^2 + sum unmatched (d - b)^2 / 2 in double.  Returns 0, or -1 (bad arguments,
 * cap too small).
 */
int to_betti_matching(const float* L, const float* G, int H, int W, int dim, int32_t* matched, int32_t* up,
                      int32_t* ut, int cap, int32_t* counts, double* cost) {
    if (H <= 0 || W <= 0 || (dim != 0 && dim != 1)) return -1;
    const int N = H * W, NN = dim == 0 ? (H + 1) * (W + 1) : H * W + 1;
    const size_t ncell = (size_t)(2 * H + 1) * (size_t)(2 * W + 1);
    float* C = (float*)malloc(sizeof(float) * (size_t)N);
    for (int k = 0; k < N; ++k) C[k] = fmin2(L[k], G[k]);
    int32_t* P[2]; int32_t* I[2]; int32_t* part[2]; int32_t* tab[2];
    const float* M[2] = {L, G};
    for (int s = 0; s < 2; ++s) {
        P[s] = (int32_t*)malloc(sizeof(int32_t) * (size_t)NN);
        I[s] = (int32_t*)malloc(sizeof(int32_t) * (size_t)NN);
        part[s] = (int32_t*)malloc(sizeof(int32_t) * (size_t)NN);
        tab[s] = (int32_t*)malloc(sizeof(int32_t) * ncell);
        for (int y = 0; y < NN; ++y) part[s][y] = -1;
        for (size_t c = 0; c < ncell; ++c) tab[s][c] = -1;
        image_kruskal(M[s], M[s], H, W, dim, P[s]);
        if (dim == 0) { image_kruskal(M[s], C, H, W, 0, I[s]); keep_positive(M[s], C, H, W, 0, I[s]); }
        else { image_kruskal(C, M[s], H, W, 1, I[s]); keep_positive(C, M[s], H, W, 1, I[s]); }
    }
    int32_t root[2] = {-1, -1};
    for (int s = 0; s < 2; ++s) {
        if (dim == 0) for (int y = 0; y < NN; ++y) if (P[s][y] < 0) root[s] = y;
        keep_positive(M[s], M[s], H, W, dim, P[s]);
    }
    if (dim == 0) {  /* death edge in C -> node of the other map's image interval */
        for (int s = 0; s < 2; ++s) for (int y = 0; y < NN; ++y) if (I[s][y] >= 0) tab[s][I[s][y]] = y;
        for (int s = 0; s < 2; ++s)
            for (int y = 0; y < NN; ++y) {
                if (P[s][y] < 0 || I[s][y] < 0) continue;
                const int32_t o = tab[1 - s][I[s][y]];
                if (o >= 0 && P[1 - s][o] >= 0) part[s][y] = o;
            }
    } else {  /* birth edge -> the barcode interval's node, then through the death square of C */
        for (int s = 0; s < 2; ++s) for (int y = 0; y < NN; ++y) if (P[s][y] >= 0) tab[s][P[s][y]] = y;
        for (int y = 0; y < NN; ++y) {
            if (I[0][y] < 0 || I[1][y] < 0) continue;
            const int32_t z = tab[0][I[0][y]], zg = tab[1][I[1][y]];
            if (z >= 0 && zg >= 0) { part[0][z] = zg; part[1][zg] = z; }
        }
    }
    int nm = 0, np_ = 0, nt = 0, rc = 0;
    double acc = 0.0;
    for (int y = 0; y < NN && rc == 0; ++y) {
        if (P[0][y] < 0) continue;
        int32_t a, b;
        interval_pixels(L, H, W, dim, y, P[0][y], &a, &b);
        if (part[0][y] >= 0) {
            int32_t c, d;
            const int32_t z = part[0][y];
            interval_pixels(G, H, W, dim, z, P[1][z], &c, &d);
            if (nm >= cap) { rc = -1; break; }
            matched[4 * nm] = a; matched[4 * nm + 1] = b; matched[4 * nm + 2] = c; matched[4 * nm + 3] = d; ++nm;
            acc += ((double)L[a] - (double)G[c]) * ((double)L[a] - (double)G[c]) + ((double)L[b] - (double)G[d]) * ((double)L[b] - (double)G[d]);
        } else {
            if (np_ >= cap) { rc = -1; break; }
            up[2 * np_] = a; up[2 * np_ + 1] = b; ++np_;
            acc += ((double)L[b] - (double)L[a]) * ((double)L[b] - (double)L[a]) / 2.0;
        }
    }
    for (int y = 0; y < NN && rc == 0; ++y) {
        if (P[1][y] < 0 || part[1][y] >= 0) continue;
        int32_t c, d;
        interval_pixels(G, H, W, dim, y, P[1][y], &c, &d);
        if (nt >= cap) { rc = -1; break; }
        ut[2 * nt] = c; ut[2 * nt + 1] = d; ++nt;
        acc += ((double)G[d] - (double)G[c]) * ((double)G[d] - (double)G[c]) / 2.0;
    }
    if (dim == 0 && rc == 0) {
        if (nm >= cap) rc = -1;
        else {
            int32_t a, c, ma = 0, mg = 0;
            vertex_val_top(L, H, W, root[0] / (W + 1), root[0] % (W + 1), &a);
            vertex_val_top(G, H, W, root[1] / (W + 1), root[1] % (W + 1), &c);
            for (int k = 1; k < N; ++k) { if (L[k] > L[ma]) ma = k; if (G[k] > G[mg]) mg = k; }
            matched[4 * nm] = a; matched[4 * nm + 1] = ma; matched[4 * nm + 2] = c; matched[4 * nm + 3] = mg; ++nm;
            acc += ((double)L[a] - (double)G[c]) * ((double)L[a] - (double)G[c]) + ((double)L[ma] - (double)G[mg]) * ((double)L[ma] - (double)G[mg]);
        }
    }
    counts[0] = nm; counts[1] = np_; counts[2] = nt;
    *cost = acc;
    for (int s = 0; s < 2; ++s) { free(P[s]); free(I[s]); free(part[s]); free(tab[s]); }
    free(C);
    return rc;
}

