/* TEST INFRASTRUCTURE -- host build of the LBVH, the bit-exact check target for the GPU builder
 * (dogeray_b200/csrc/scene.cu).  The reference has no LBVH (its build_bvh, kernel.cu:1864-1909, is a
 * host median split, restated in dogeray_oracle.c); this file restates the PRODUCT's build steps in
 * scalar C so that its integer outputs -- Morton keys, sorted order, Karras topology -- and the
 * refitted boxes can be compared with what the device produced, bit for bit.
 *
 * Steps (same single IEEE operations as the device code; compile with -ffp-contract=off):
 *   scene bounds = min / max over primitive boxes
 *   key = 63-bit Morton code of the box centre ((lo + hi) * 0.5), 21 bits per axis, x most significant,
 *         axis value = (uint)clamp(((c - slo) / ext) * 2097152, 0, 2097151), ext = shi - slo or 1 if not > 0
 *   stable sort of (key, slot)
 *   Karras 2012 hierarchy, delta(i, j) = clz64(key_i ^ key_j), or 64 + clz32(i ^ j) when the keys tie
 *   bottom-up box union
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

static uint64_t spread21(uint32_t v)
{
    uint64_t x = v & 0x1FFFFFull;
    x = (x | (x << 32)) & 0x1F00000000FFFFull;
    x = (x | (x << 16)) & 0x1F0000FF0000FFull;
    x = (x | (x << 8)) & 0x100F00F00F00F00Full;
    x = (x | (x << 4)) & 0x10C30C30C30C30C3ull;
    x = (x | (x << 2)) & 0x1249249249249249ull;
    return x;
}

typedef struct { uint64_t key; int32_t slot; } kv;
static int kv_cmp(const void* a, const void* b)
{
    const kv* p = (const kv*)a; const kv* q = (const kv*)b;
    if (p->key != q->key) return p->key < q->key ? -1 : 1;
    return (p->slot > q->slot) - (p->slot < q->slot);          /* = stable order of the radix sort */
}

static int delta(const uint64_t* keys, int n, int i, int j)
{
    if (j < 0 || j >= n) return -1;
    uint64_t a = keys[i], b = keys[j];
    if (a != b) return __builtin_clzll(a ^ b);
    return 64 + __builtin_clz((unsigned)(i ^ j));
}

static void node_box(int c, const float* lmin, const float* lmax, const float* nmin, const float* nmax, float lo[3], float hi[3])
{
    const float* a = c < 0 ? lmin + 3 * (size_t)(~c) : nmin + 3 * (size_t)c;
    const float* b = c < 0 ? lmax + 3 * (size_t)(~c) : nmax + 3 * (size_t)c;
    memcpy(lo, a, 12); memcpy(hi, b, 12);
}

/* bmin/bmax: n*3 primitive boxes in slot order.  Outputs as drb_scene_lbvh: keys[n] and order[n] sorted;
 * parent/left/right[n-1]; node_min/node_max[(n-1)*3]; scene_bounds[6].  Returns the tree height. */
int lbvh_host_build(const float* bmin, const float* bmax, int n, uint64_t* keys, int32_t* order, int32_t* parent, int32_t* left,
                    int32_t* right, float* node_min, float* node_max, float* scene_bounds)
{
    if (n <= 0) return 0;
    float slo[3] = { bmin[0], bmin[1], bmin[2] }, shi[3] = { bmax[0], bmax[1], bmax[2] };
    for (int i = 1; i < n; i++)
        for (int a = 0; a < 3; a++) {
            if (bmin[3 * i + a] < slo[a]) slo[a] = bmin[3 * i + a];
            if (bmax[3 * i + a] > shi[a]) shi[a] = bmax[3 * i + a];
        }
    if (scene_bounds) { memcpy(scene_bounds, slo, 12); memcpy(scene_bounds + 3, shi, 12); }
    kv* tmp = (kv*)malloc(sizeof(kv) * (size_t)n);
    for (int i = 0; i < n; i++) {
        uint32_t q[3];
        for (int a = 0; a < 3; a++) {
            float c = (bmin[3 * i + a] + bmax[3 * i + a]) * 0.5f;
            float ext = shi[a] - slo[a];
            if (!(ext > 0.0f)) ext = 1.0f;
            float x = ((c - slo[a]) / ext) * 2097152.0f;
            x = fminf(fmaxf(x, 0.0f), 2097151.0f);
            q[a] = (uint32_t)x;
        }
        tmp[i].key = (spread21(q[0]) << 2) | (spread21(q[1]) << 1) | spread21(q[2]);
        tmp[i].slot = i;
    }
    qsort(tmp, (size_t)n, sizeof(kv), kv_cmp);
    for (int i = 0; i < n; i++) { keys[i] = tmp[i].key; order[i] = tmp[i].slot; }
    free(tmp);
    if (n == 1) return 1;

    int32_t* leaf_parent = (int32_t*)malloc(sizeof(int32_t) * (size_t)n);
    for (int i = 0; i < n - 1; i++) {
        int d = (delta(keys, n, i, i + 1) - delta(keys, n, i, i - 1)) >= 0 ? 1 : -1;
        int dmin = delta(keys, n, i, i - d);
        int lmax = 2;
        while (delta(keys, n, i, i + lmax * d) > dmin) lmax <<= 1;
        int l = 0;
        for (int t = lmax >> 1; t >= 1; t >>= 1)
            if (delta(keys, n, i, i + (l + t) * d) > dmin) l += t;
        int j = i + l * d;
        int dnode = delta(keys, n, i, j);
        int s = 0;
        for (int t = (l + 1) >> 1;; t = (t + 1) >> 1) {
            if (delta(keys, n, i, i + (s + t) * d) > dnode) s += t;
            if (t <= 1) break;
        }
        int gamma = i + s * d + (d < 0 ? d : 0);
        int lo = i < j ? i : j, hi = i < j ? j : i;
        int lc = (lo == gamma) ? ~gamma : gamma;
        int rc = (hi == gamma + 1) ? ~(gamma + 1) : gamma + 1;
        left[i] = lc; right[i] = rc;
        if (lc < 0) leaf_parent[gamma] = i; else parent[gamma] = i;
        if (rc < 0) leaf_parent[gamma + 1] = i; else parent[gamma + 1] = i;
    }
    parent[0] = -1;

    /* leaf boxes in sorted order */
    float* lmin = (float*)malloc(12 * (size_t)n); float* lmax = (float*)malloc(12 * (size_t)n);
    for (int k = 0; k < n; k++) { memcpy(lmin + 3 * k, bmin + 3 * (size_t)order[k], 12); memcpy(lmax + 3 * k, bmax + 3 * (size_t)order[k], 12); }
    /* bottom-up: a node is ready when both children are; process by repeated leaf climbs like the device */
    int* visits = (int*)calloc((size_t)(n - 1), sizeof(int));
    int* height = (int*)calloc((size_t)(n - 1), sizeof(int));
    int tree_height = 0;
    for (int k = 0; k < n; k++) {
        int node = leaf_parent[k];
        while (node >= 0) {
            if (visits[node]++ == 0) break;
            float a0[3], a1[3], b0[3], b1[3];
            node_box(left[node], lmin, lmax, node_min, node_max, a0, a1);
            node_box(right[node], lmin, lmax, node_min, node_max, b0, b1);
            for (int a = 0; a < 3; a++) { node_min[3 * node + a] = fminf(a0[a], b0[a]); node_max[3 * node + a] = fmaxf(a1[a], b1[a]); }
            int hl = left[node] < 0 ? 0 : height[left[node]], hr = right[node] < 0 ? 0 : height[right[node]];
            height[node] = (hl > hr ? hl : hr) + 1;
            if (node == 0) tree_height = height[0];
            node = parent[node];
        }
    }
    free(visits); free(height); free(lmin); free(lmax); free(leaf_parent);
    return tree_height;
}

/* ---- host mirror of the SAH-guided rebuild (k_ploc_* in dogeray_b200/csrc/scene.cu) ----------------
 * lmin/lmax: n*3 leaf boxes in SORTED order.  Outputs in the final labelling (root = node 0): left/right
 * [n-1] with leaves as ~sorted_position, node_min/node_max [(n-1)*3].  Returns the tree height; *rounds gets the
 * number of clustering rounds (drb_build_info.rebuild_iterations of the device build). */
static float union_half_area(const float* alo, const float* ahi, const float* blo, const float* bhi)
{
    float ex = fmaxf(ahi[0], bhi[0]) - fminf(alo[0], blo[0]);
    float ey = fmaxf(ahi[1], bhi[1]) - fminf(alo[1], blo[1]);
    float ez = fmaxf(ahi[2], bhi[2]) - fminf(alo[2], blo[2]);
    return ex * ey + ey * ez + ez * ex;
}

int ploc_host_build(const float* lmin, const float* lmax, int n, int radius, int32_t* left, int32_t* right, float* node_min, float* node_max,
                    int* rounds)
{
    *rounds = 0;
    if (n <= 1) return n;
    size_t N = (size_t)n;
    int32_t* cid[2]; float* cmn[2]; float* cmx[2]; int* chg[2];
    for (int k = 0; k < 2; k++) { cid[k] = malloc(4 * N); cmn[k] = malloc(12 * N); cmx[k] = malloc(12 * N); chg[k] = malloc(4 * N); }
    int32_t* nn = malloc(4 * N);
    int32_t* pl = malloc(4 * N); int32_t* pr = malloc(4 * N); float* pmin = malloc(12 * N); float* pmax = malloc(12 * N);
    for (int i = 0; i < n; i++) { cid[0][i] = ~i; chg[0][i] = 0; }
    memcpy(cmn[0], lmin, 12 * N); memcpy(cmx[0], lmax, 12 * N);
    int cur = 0, m = n, node_base = 0, height = 0;
    while (m > 1) {
        for (int i = 0; i < m; i++) {
            float best = 3.4e38f; int bj = -1;
            int j0 = i - radius < 0 ? 0 : i - radius, j1 = i + radius > m - 1 ? m - 1 : i + radius;
            for (int j = j0; j <= j1; j++) {
                if (j == i) continue;
                float a = union_half_area(cmn[cur] + 3 * i, cmx[cur] + 3 * i, cmn[cur] + 3 * j, cmx[cur] + 3 * j);
                const int d = abs(i - j), bd = abs(i - bj);
                if (a < best || (a == best && (d < bd || (d == bd && (i ^ j) < (i ^ bj))))) { best = a; bj = j; }
            }
            if (bj < 0) bj = (i ^ 1) < m ? (i ^ 1) : i - 1;
            nn[i] = bj;
        }
        int pos = 0, merges = 0, nx = cur ^ 1;
        ++*rounds;
        for (int i = 0; i < m; i++) {
            int j = nn[i];
            int mutual = j >= 0 && j < m && nn[j] == i;
            if (mutual && i > j) continue;
            if (mutual && i < j) {
                int node = node_base + merges++;
                pl[node] = cid[cur][i]; pr[node] = cid[cur][j];
                for (int a = 0; a < 3; a++) {
                    pmin[3 * node + a] = fminf(cmn[cur][3 * i + a], cmn[cur][3 * j + a]);
                    pmax[3 * node + a] = fmaxf(cmx[cur][3 * i + a], cmx[cur][3 * j + a]);
                }
                int h = (chg[cur][i] > chg[cur][j] ? chg[cur][i] : chg[cur][j]) + 1;
                cid[nx][pos] = node; chg[nx][pos] = h; height = h;
                memcpy(cmn[nx] + 3 * pos, pmin + 3 * node, 12); memcpy(cmx[nx] + 3 * pos, pmax + 3 * node, 12);
            } else {
                cid[nx][pos] = cid[cur][i]; chg[nx][pos] = chg[cur][i];
                memcpy(cmn[nx] + 3 * pos, cmn[cur] + 3 * i, 12); memcpy(cmx[nx] + 3 * pos, cmx[cur] + 3 * i, 12);
            }
            pos++;
        }
        if (merges == 0) break;
        node_base += merges; m = pos; cur = nx;
    }
    height = chg[cur][0];
    for (int i = 0; i < n - 1; i++) {
        int dst = (n - 2) - i;
        left[dst] = pl[i] < 0 ? pl[i] : (n - 2) - pl[i];
        right[dst] = pr[i] < 0 ? pr[i] : (n - 2) - pr[i];
        memcpy(node_min + 3 * dst, pmin + 3 * i, 12); memcpy(node_max + 3 * dst, pmax + 3 * i, 12);
    }
    for (int k = 0; k < 2; k++) { free(cid[k]); free(cmn[k]); free(cmx[k]); free(chg[k]); }
    free(nn); free(pl); free(pr); free(pmin); free(pmax);
    return height;
}

/* ---- host mirror of the four-wide collapse (k_wide_* in dogeray_b200/csrc/scene.cu) ---------------------
 * Input: the final binary tree (root 0; left/right with leaves as ~sorted_position; node boxes; sorted leaf
 * boxes) and the scene bounds.  Output: child[4*i + k], boxes[12*i + 3*k + a] (min_q | max_q << 16 on the
 * 16-bit scene grid), breadth-first ids.  Returns the number of wide nodes; *levels gets the tree height. */
static float box_half_area3(const float* lo, const float* hi)
{
    float ex = hi[0] - lo[0], ey = hi[1] - lo[1], ez = hi[2] - lo[2];
    return ex * ey + ey * ez + ez * ex;
}
static uint32_t quant_axis_h(float lo, float hi, float qlo, float qscale)
{
    int a = (int)floorf((lo - qlo) / qscale) - 1;
    int b = (int)ceilf((hi - qlo) / qscale) + 1;
    if (a < 0) a = 0;
    if (a > 65535) a = 65535;
    if (b < 0) b = 0;
    if (b > 65535) b = 65535;
    return (uint32_t)a | ((uint32_t)b << 16);
}
#define WIDE_EMPTY ((int32_t)0x80000000)

int wide_host_build(const int32_t* left, const int32_t* right, const float* node_min, const float* node_max, const float* lmin,
                    const float* lmax, int n, const float* scene_bounds, int32_t* child, uint32_t* boxes, int* levels)
{
    float qlo[3], qs[3];
    for (int a = 0; a < 3; a++) {
        float ext = scene_bounds[3 + a] - scene_bounds[a];
        if (!(ext > 0.0f)) ext = 1.0f;
        qs[a] = ext / 65527.0f;
        qlo[a] = scene_bounds[a] - 4.0f * qs[a];
    }
    if (n == 1) {
        for (int k = 0; k < 4; k++) { child[k] = WIDE_EMPTY; for (int a = 0; a < 3; a++) boxes[3 * k + a] = 0x0000FFFFu; }
        child[0] = ~0;
        for (int a = 0; a < 3; a++) boxes[a] = quant_axis_h(lmin[a], lmax[a], qlo[a], qs[a]);
        *levels = 1;
        return 1;
    }
    int32_t* q[2]; q[0] = malloc(4 * (size_t)n); q[1] = malloc(4 * (size_t)n);
    q[0][0] = 0;
    int nq = 1, base = 0, cur = 0, lev = 0;
    while (nq > 0) {
        int next = 0, next_base = base + nq;
        for (int i = 0; i < nq; i++) {
            int b = q[cur][i];
            int s[4] = { left[b], right[b], WIDE_EMPTY, WIDE_EMPTY };
            int cnt = 2;
            for (int it = 0; it < 2; it++) {
                int pick = -1; float best = -1.0f;
                for (int k = 0; k < cnt; k++)
                    if (s[k] >= 0) {
                        float ar = box_half_area3(node_min + 3 * (size_t)s[k], node_max + 3 * (size_t)s[k]);
                        if (ar > best) { best = ar; pick = k; }
                    }
                if (pick < 0) break;
                int c = s[pick];
                s[pick] = left[c];
                s[cnt++] = right[c];
            }
            int id = base + i;
            for (int k = 0; k < 4; k++) {
                int link = WIDE_EMPTY;
                uint32_t qq[3] = { 0x0000FFFFu, 0x0000FFFFu, 0x0000FFFFu };
                if (s[k] != WIDE_EMPTY) {
                    const float* lo = s[k] < 0 ? lmin + 3 * (size_t)(~s[k]) : node_min + 3 * (size_t)s[k];
                    const float* hi = s[k] < 0 ? lmax + 3 * (size_t)(~s[k]) : node_max + 3 * (size_t)s[k];
                    for (int a = 0; a < 3; a++) qq[a] = quant_axis_h(lo[a], hi[a], qlo[a], qs[a]);
                    if (s[k] < 0) link = s[k];
                    else { link = next_base + next; q[cur ^ 1][next++] = s[k]; }
                }
                child[4 * (size_t)id + k] = link;
                for (int a = 0; a < 3; a++) boxes[12 * (size_t)id + 3 * k + a] = qq[a];
            }
        }
        base = next_base; nq = next; cur ^= 1; lev++;
    }
    free(q[0]); free(q[1]);
    *levels = lev;
    return base;
}
