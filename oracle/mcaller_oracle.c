/*
 * mcaller_oracle.c -- CPU restatement of the mCaller hot path.  TEST INFRASTRUCTURE ONLY.
 *
 * This file is the checker the CUDA path is compared against.  It may be imported / linked /
 * executed only from tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
 * legs.  It is never a fallback for the product path (mcaller_b200 fails loudly without its CUDA
 * library).
 *
 * Parity status: PINNED.  tests/test_oracle_golden.py checks this restatement against
 *   (a) the reference's own fixtures (testdata/masonread1.*: 9-row .diffs.6 feature block, 44-row
 *       .diffs.6.train windows, 5-row BED), and
 *   (b) outputs of the unmodified reference run in the build container on 17 deterministic inputs
 *       (tools/make_golden.py -> tests/golden/*.json): rows, feature text, probabilities text,
 *       labels, the five stdout counters, BED rows.
 *
 * What it follows (file:line into the reference, al-mcintyre/mCaller):
 *   extract_contexts.py:140-152  line reader + whitespace tokeniser        -> next_line / split_ws
 *   extract_contexts.py:154-176  contig / first_read_ind / quality / strand -> orc_extract main loop
 *   extract_contexts.py:179-266  window close, skip filter, multi-M carry   -> close_window
 *   extract_contexts.py:269-291  feed / reset                               -> feed part of the loop
 *   extract_contexts.py:99-106   base_models                                -> select_model
 *   extract_contexts.py:195-207  classifier call + label                    -> orc_predict
 *   make_bed.py:21-28, 67-98, 132-159  per-position aggregation             -> orc_aggregate
 * Third-party arithmetic restated from published behaviour (not under /root/reference):
 *   numpy add.reduce pairwise summation (np.mean, :186)  -> np_mean  (checked against numpy 2.3.5)
 *   numpy round (np.round(x,4), :286)                   -> np_round4
 *   scikit-learn MLPClassifier._forward_pass_fast / LogisticRegression / GaussianNB /
 *   RandomForestClassifier.predict_proba (1.9.0)        -> orc_predict
 *
 * Deliberate, documented deviations: '\r' is treated as intra-line whitespace (the reference, in
 * text mode, would hang on CR-containing files because its character count never reaches the byte
 * size, :144-148); fatal paths of the reference (print + sys.exit(0)) return negative error codes.
 */
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#define ORC_MAXK 16

typedef struct {
    const char *name;     /* contig id */
    const char *fwd;      /* forward-strand marked copy ('M' at targets) */
    const char *rev;      /* reverse-strand marked copy, forward coordinates */
    int64_t len;
} orc_contig;

typedef struct {
    const char *key;      /* read-name prefix (FASTQ id up to first ':' / '_') */
    double qual;
} orc_qual;               /* table sorted by strcmp(key) */

enum { ORC_MLP = 0, ORC_LR = 1, ORC_GNB = 2, ORC_RF = 3 };
enum { ACT_IDENTITY = 0, ACT_LOGISTIC = 1, ACT_TANH = 2, ACT_RELU = 3 };

typedef struct {
    int32_t kind;
    int32_t n_in;
    /* MLP: n_layers weight matrices; layer l has shape [sizes[l], sizes[l+1]] row-major (sklearn coefs_[l]) */
    int32_t n_layers;
    int32_t sizes[8];
    int32_t hidden_act;
    const double *weights;   /* concatenated coefs_ */
    const double *biases;    /* concatenated intercepts_ */
    /* LR: weights[n_in], biases[1].  GNB: weights = theta[2][n_in] then var[2][n_in]; biases = log prior[2] */
    /* RF: flat node arrays over all trees */
    int32_t n_trees;
    const int32_t *tree_off;     /* [n_trees+1] node offsets */
    const int32_t *left;         /* -1 for leaf */
    const int32_t *right;
    const int32_t *feature;
    const double *threshold;
    const double *leaf_p1;       /* per node: class-1 fraction of node value */
} orc_model;

typedef struct {
    int32_t kind;            /* 0 = emitted call, 1 = too-many-skips event, 2 = multi-M event */
    int32_t chrom_cid;       /* contig of the CLOSING line (column 1, reference :216) */
    int32_t win_cid;         /* contig the window lies on (last_ref) */
    int32_t rev;             /* last_rev */
    int64_t read_off;        /* last_read: offset/len of the name inside the text buffer */
    int32_t read_len;
    int32_t mpos;
    int32_t n_empty;
    uint32_t empty_mask;     /* bit c set: output feature c printed as integer 0 (empty column) */
    int32_t model_sel;       /* 0 = 'general' or 'MH', 1 = 'MG' */
    int32_t label;           /* 1 if prob >= 0.5 */
    double feat[ORC_MAXK + 1];   /* k features in output order + read quality */
    double prob;
    char context[2 * ORC_MAXK];  /* 2k-1 chars + NUL */
} orc_call;

typedef struct {
    double *v;
    int n, cap;
} col_t;

/* ---- numpy restatements ------------------------------------------------------------------- */

/* numpy/_core/src/umath/loops_utils.h.src  @TYPE@_pairwise_sum, as reached from add.reduce on a
 * contiguous float64 array (np.mean of a list, extract_contexts.py:186). */
static double np_pairwise(const double *a, int64_t n) {
    if (n < 8) {
        double res = 0.;
        for (int64_t i = 0; i < n; i++) res += a[i];
        return res;
    } else if (n <= 128) {
        double r[8];
        int64_t i;
        for (i = 0; i < 8; i++) r[i] = a[i];
        for (i = 8; i < n - (n % 8); i += 8)
            for (int j = 0; j < 8; j++) r[j] += a[i + j];
        double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
        for (; i < n; i++) res += a[i];
        return res;
    } else {
        int64_t n2 = n / 2;
        n2 -= n2 % 8;
        return np_pairwise(a, n2) + np_pairwise(a + n2, n - n2);
    }
}

/* add.reduce adds the pairwise sum to its initial 0.0, so a sum of -0.0 values comes out as 0.0 */
double orc_np_mean(const double *a, int64_t n) { return (np_pairwise(a, n) + 0.0) / (double)n; }

/* np.round(x, 4): multiply, rint, divide (numpy/_core/src/multiarray/calculation.c PyArray_Round) */
double orc_np_round(double x, int decimals) {
    double f = 1.0;
    for (int i = 0; i < decimals; i++) f *= 10.0;
    return rint(x * f) / f;
}

/* ---- small helpers ------------------------------------------------------------------------ */

static int is_ws(unsigned char c) {
    /* str.split() whitespace for ASCII text; '\n' never reaches here (line terminator) */
    return c == ' ' || (c >= 9 && c <= 13) || (c >= 28 && c <= 31);
}

typedef struct { const char *p; int len; } tok_t;

static int tok_eq(tok_t a, tok_t b) { return a.len == b.len && memcmp(a.p, b.p, (size_t)a.len) == 0; }
static int tok_is(tok_t a, const char *s) { return (int)strlen(s) == a.len && memcmp(a.p, s, (size_t)a.len) == 0; }

static int split_ws(const char *p, const char *end, tok_t *f, int maxf) {
    int n = 0;
    while (p < end) {
        while (p < end && is_ws((unsigned char)*p)) p++;
        if (p >= end) break;
        const char *s = p;
        while (p < end && !is_ws((unsigned char)*p)) p++;
        if (n < maxf) { f[n].p = s; f[n].len = (int)(p - s); }
        n++;
        if (n >= maxf) break;   /* line.split()[:12] -- only the count up to 12 matters */
    }
    return n;
}

static int parse_i64(tok_t t, int64_t *out) {
    char buf[64];
    if (t.len <= 0 || t.len >= 63) return -1;
    memcpy(buf, t.p, (size_t)t.len); buf[t.len] = 0;
    char *e; long long v = strtoll(buf, &e, 10);
    if (*e) return -1;
    *out = v; return 0;
}

static int parse_f64(tok_t t, double *out) {
    char buf[128];
    if (t.len <= 0 || t.len >= 127) return -1;
    memcpy(buf, t.p, (size_t)t.len); buf[t.len] = 0;
    char *e; double v = strtod(buf, &e);
    if (*e) return -1;
    *out = v; return 0;
}

static int qual_lookup(const orc_qual *q, int64_t nq, const char *name, int len, double *out) {
    /* read2qual[name] else read2qual[name.split(':')[0].split('_')[0]] (reference :163-166).  Keys never
     * contain ':' or '_' (read_qual.py:11-12), so both lookups reduce to the prefix lookup. */
    int plen = 0;
    while (plen < len && name[plen] != ':' && name[plen] != '_') plen++;
    int64_t lo = 0, hi = nq - 1;
    while (lo <= hi) {
        int64_t mid = (lo + hi) / 2;
        int c = strncmp(q[mid].key, name, (size_t)plen);
        if (c == 0) c = (q[mid].key[plen] == 0) ? 0 : 1;
        if (c == 0) { *out = q[mid].qual; return 0; }
        if (c < 0) lo = mid + 1; else hi = mid - 1;
    }
    return -1;
}

static void col_push(col_t *c, double v) {
    if (c->n == c->cap) { c->cap = c->cap ? 2 * c->cap : 8; c->v = (double *)realloc(c->v, sizeof(double) * (size_t)c->cap); }
    c->v[c->n++] = v;
}

static char comp_char(char c) {
    switch (c) { case 'A': return 'T'; case 'C': return 'G'; case 'G': return 'C'; case 'T': return 'A'; case 'N': return 'N'; case 'M': return 'M'; }
    return 0;   /* KeyError in the reference */
}

/* ---- classifier ----------------------------------------------------------------------------- */

static double expit(double x) { return x < 0 ? exp(x) / (1.0 + exp(x)) : 1.0 / (1.0 + exp(-x)); }

double orc_predict(const orc_model *m, const double *x) {
    if (m->kind == ORC_MLP) {
        double a[512], b[512];
        const double *w = m->weights, *bi = m->biases;
        for (int i = 0; i < m->sizes[0]; i++) a[i] = x[i];
        for (int l = 0; l < m->n_layers; l++) {
            int ni = m->sizes[l], no = m->sizes[l + 1];
            for (int o = 0; o < no; o++) {
                double acc = 0.0;
                for (int i = 0; i < ni; i++) acc += a[i] * w[(size_t)i * no + o];
                acc += bi[o];
                if (l + 1 < m->n_layers) {
                    switch (m->hidden_act) {
                        case ACT_TANH: acc = tanh(acc); break;
                        case ACT_LOGISTIC: acc = expit(acc); break;
                        case ACT_RELU: acc = acc > 0 ? acc : 0; break;
                        default: break;
                    }
                }
                b[o] = acc;
            }
            memcpy(a, b, sizeof(double) * (size_t)no);
            w += (size_t)ni * no; bi += no;
        }
        return expit(a[0]);
    } else if (m->kind == ORC_LR) {
        double z = m->biases[0];
        for (int i = 0; i < m->n_in; i++) z += x[i] * m->weights[i];
        return expit(z);
    } else if (m->kind == ORC_GNB) {
        /* sklearn naive_bayes.py GaussianNB._joint_log_likelihood + predict_proba */
        const double *theta = m->weights, *var = m->weights + 2 * m->n_in;
        double jll[2];
        for (int c = 0; c < 2; c++) {
            double n_ij = 0.0, s = 0.0;
            for (int i = 0; i < m->n_in; i++) n_ij += log(2.0 * M_PI * var[c * m->n_in + i]);
            n_ij *= -0.5;
            for (int i = 0; i < m->n_in; i++) { double d = x[i] - theta[c * m->n_in + i]; s += d * d / var[c * m->n_in + i]; }
            jll[c] = m->biases[c] + n_ij - 0.5 * s;
        }
        double mx = jll[0] > jll[1] ? jll[0] : jll[1];
        double lse = mx + log(exp(jll[0] - mx) + exp(jll[1] - mx));
        return exp(jll[1] - lse);
    } else {
        /* sklearn ensemble/_forest.py predict_proba: mean over trees of the leaf class fractions;
         * the tree walk compares float32(x) <= threshold (tree/_tree.pyx) */
        double acc = 0.0;
        for (int t = 0; t < m->n_trees; t++) {
            int32_t n = m->tree_off[t];
            while (m->left[n] >= 0) {
                float xv = (float)x[m->feature[n]];
                n = ((double)xv <= m->threshold[n]) ? m->tree_off[t] + m->left[n] : m->tree_off[t] + m->right[n];
            }
            acc += m->leaf_p1[n];
        }
        return acc / m->n_trees;
    }
}

/* ---- extract_features ------------------------------------------------------------------------ */

typedef struct {
    orc_call *calls; int64_t n, cap;
} out_t;

static orc_call *out_next(out_t *o) {
    if (o->n >= o->cap) return NULL;
    orc_call *c = &o->calls[o->n++];
    memset(c, 0, sizeof(*c));
    return c;
}

#define ERR_CAP -2
#define ERR_QUAL_KEY -3
#define ERR_NUMERIC -4
#define ERR_CONTEXT -5
#define ERR_MODEL_KEY -6
#define ERR_NDIFFS -7

/*
 * two_models: 1 when the pickle is a dict with 'MG'/'MH' and base == 'A' (reference :126-131, :100-101);
 * models[0] = 'MH' or 'general', models[1] = 'MG'.
 * Returns number of records written to calls (kinds 0/1/2 interleaved in event order) or <0 on error.
 */
int64_t orc_extract(const char *text, int64_t nbytes,
                    const orc_contig *contigs, int32_t n_contigs,
                    const orc_qual *quals, int64_t n_quals,
                    int32_t k, int32_t skip_thresh, double qual_thresh,
                    const orc_model *models, int32_t two_models, int32_t do_predict,
                    orc_call *calls, int64_t cap)
{
    out_t out = { calls, 0, cap };
    col_t col[ORC_MAXK]; memset(col, 0, sizeof(col));
    col_t tmpc[ORC_MAXK];
    int64_t rc = 0;

    tok_t last_read = { "", 0 };
    int last_contig = -1;                 /* None */
    int has_mpos = 0; int64_t mpos = 0;   /* Python: mpos = None */
#define MPOS_TRUTHY (has_mpos && mpos != 0)
    int64_t first_read_ind = 0;
    int last_rev = 0, last_cid = -1;
    const char *meth_fwd = NULL, *meth_rev = NULL; int64_t clen = 0;

    const char *p = text, *end = text + nbytes;
    while (p < end) {
        const char *nl = (const char *)memchr(p, '\n', (size_t)(end - p));
        const char *le = nl ? nl : end;
        tok_t f[12];
        int nf = split_ws(p, le, f, 12);
        p = nl ? nl + 1 : end;
        if (nf < 12) continue;                                              /* :149-152 */
        tok_t chrom = f[0], read_pos_t = f[1], read_kmer = f[2], read_name = f[3], read_ind_t = f[5],
              ev_t = f[6], ref_kmer = f[9], model_t = f[10];

        if (last_contig < 0 || !tok_is(chrom, contigs[last_contig].name)) {   /* :154-160 */
            int found = -1;
            for (int c = 0; c < n_contigs; c++) if (tok_is(chrom, contigs[c].name)) { found = c; break; }
            if (found < 0) continue;
            last_contig = found;
            meth_fwd = contigs[found].fwd; meth_rev = contigs[found].rev; clen = contigs[found].len;
        }
        int same_read = tok_eq(read_name, last_read);
        int64_t read_ind = 0;
        if (!same_read) {                                                    /* :161-162 */
            if (parse_i64(read_ind_t, &read_ind)) { rc = ERR_NUMERIC; goto done; }
            first_read_ind = read_ind;
        }
        double qual;
        if (qual_lookup(quals, n_quals, read_name.p, read_name.len, &qual)) { rc = ERR_QUAL_KEY; goto done; }   /* :163-166 */
        if (qual < qual_thresh || tok_is(ref_kmer, "NNNNNN")) continue;      /* :167-168 */
        int rev;
        if (!same_read) rev = !tok_eq(read_kmer, ref_kmer);                  /* :169-174 */
        else {
            if (parse_i64(read_ind_t, &read_ind)) { rc = ERR_NUMERIC; goto done; }
            rev = !(read_ind > first_read_ind);
        }
        const char *meth_ref = rev ? meth_rev : meth_fwd;
        int64_t read_pos;
        if (parse_i64(read_pos_t, &read_pos) || read_pos < 0) { rc = ERR_NUMERIC; goto done; }   /* :175 */
        /* reference_kmer = meth_ref[read_pos:read_pos+k] (:176), Python slice clamps at the end */
        int klen = 0; int first_m = -1;
        for (int i = 0; i < k && read_pos + i < clen; i++) { klen++; if (meth_ref[read_pos + i] == 'M' && first_m < 0) first_m = i; }

        if (MPOS_TRUTHY && ((read_pos >= mpos + 1 && same_read) || !same_read)) {   /* :179 */
            int num_skips = 0;
            for (int c = 0; c < k; c++) if (col[c].n == 0) num_skips++;
            if (num_skips <= skip_thresh) {                                  /* :183 */
                orc_call *oc = out_next(&out);
                if (!oc) { rc = ERR_CAP; goto done; }
                oc->kind = 0; oc->chrom_cid = last_contig; oc->win_cid = last_cid; oc->rev = last_rev;
                oc->read_off = last_read.p - text; oc->read_len = last_read.len; oc->mpos = (int32_t)mpos;
                oc->n_empty = num_skips;
                for (int c = 0; c < k; c++) {                                /* :186-188 */
                    int src = last_rev ? c : (k - 1 - c);
                    if (col[src].n == 0) { oc->feat[c] = 0.0; oc->empty_mask |= 1u << c; }
                    else oc->feat[c] = orc_np_mean(col[src].v, col[src].n);
                }
                double lq;
                if (qual_lookup(quals, n_quals, last_read.p, last_read.len, &lq)) { rc = ERR_QUAL_KEY; goto done; }
                oc->feat[k] = lq;                                            /* :189-193 */
                /* context = revcomp(last_ref[mpos-k+1:mpos+k], last_rev) (:194) */
                const orc_contig *wc = &contigs[last_cid];
                const char *lref = last_rev ? wc->rev : wc->fwd;
                int64_t a = mpos - k + 1, b = mpos + k;
                if (a < 0 || b > wc->len) { rc = ERR_CONTEXT; goto done; }
                int cl = (int)(b - a);
                for (int i = 0; i < cl; i++) {
                    char ch = last_rev ? comp_char(lref[b - 1 - i]) : lref[a + i];
                    if (!ch) { rc = ERR_CONTEXT; goto done; }
                    oc->context[i] = ch;
                }
                oc->context[cl] = 0;
                if (oc->context[cl / 2] != 'M') { rc = ERR_CONTEXT; goto done; }   /* :195, :224-228 */
                char nextb = oc->context[cl / 2 + 1];                        /* :197, base_models :99-106 */
                if (!(nextb == 'A' || nextb == 'C' || nextb == 'G' || nextb == 'T' || nextb == 'M')) { rc = ERR_MODEL_KEY; goto done; }
                oc->model_sel = (two_models && nextb == 'G') ? 1 : 0;
                if (do_predict) {
                    oc->prob = orc_predict(&models[oc->model_sel], oc->feat);   /* :199 */
                    oc->label = oc->prob >= 0.5;                             /* :200 */
                }
            } else {                                                         /* :238-239 */
                orc_call *oc = out_next(&out);
                if (!oc) { rc = ERR_CAP; goto done; }
                oc->kind = 1; oc->read_off = last_read.p - text; oc->read_len = last_read.len; oc->mpos = (int32_t)mpos;
                oc->win_cid = last_cid; oc->rev = last_rev; oc->n_empty = num_skips;
            }
            if (first_m < 0 || !same_read || read_pos > mpos + skip_thresh + 1) {   /* :242-245 */
                for (int c = 0; c < k; c++) col[c].n = 0;
                has_mpos = 0;
            } else {                                                         /* :246-256 multi-M carry */
                if (first_m != 0) {
                    orc_call *oc = out_next(&out);
                    if (!oc) { rc = ERR_CAP; goto done; }
                    oc->kind = 2; oc->read_off = last_read.p - text; oc->read_len = last_read.len; oc->mpos = (int32_t)mpos;
                    oc->win_cid = last_cid; oc->rev = last_rev;
                }
                int64_t last_mpos = mpos;
                mpos = read_pos + first_m;
                int64_t sp = mpos - last_mpos; if (sp > k) sp = k;
                if (sp <= 0) { rc = ERR_NDIFFS; goto done; }
                /* diff_col = [[]]*sp + diff_col[:-sp] */
                memcpy(tmpc, col, sizeof(col));
                for (int c = 0; c < k; c++) {
                    if (c < sp) { col[c] = tmpc[k - sp + c]; col[c].n = 0; }   /* recycle storage of dropped columns */
                    else col[c] = tmpc[c - sp];
                }
            }
        }

        if (first_m >= 0) {                                                  /* :269-287 */
            if (MPOS_TRUTHY) {
                if (!same_read) { has_mpos = 0; for (int c = 0; c < k; c++) col[c].n = 0; }
                else if (rev != last_rev) has_mpos = 0;                      /* columns NOT cleared (:276-277) */
            }
            if (!MPOS_TRUTHY) { has_mpos = 1; mpos = read_pos + first_m; }
            last_read = read_name; last_rev = rev; last_cid = last_contig;
            double ev, md;
            if (parse_f64(ev_t, &ev) || parse_f64(model_t, &md)) { rc = ERR_NUMERIC; goto done; }
            col_push(&col[first_m], orc_np_round(ev - md, 4));               /* :286 */
        } else if (MPOS_TRUTHY) {                                            /* :289-291 */
            has_mpos = 0;
            for (int c = 0; c < k; c++) col[c].n = 0;
        }
    }
    rc = out.n;
done:
    for (int c = 0; c < ORC_MAXK; c++) free(col[c].v);
    return rc;
}

int32_t orc_sizeof_call(void) { return (int32_t)sizeof(orc_call); }

/* ---- make_bed aggregate_by_pos (default mode: no -p / --gff / --vo / --ref / --plot) ----------- */

typedef struct {
    int64_t key_off[5];     /* offsets into the diffs text: csome, pos, context, strand (nextpos derived) */
    int32_t key_len[5];
    int64_t depth, meth;
} orc_locus;

static uint64_t fnv(const char *p, int n, uint64_t h) {
    for (int i = 0; i < n; i++) { h ^= (unsigned char)p[i]; h *= 1099511628211ULL; }
    return h;
}

/*
 * text: contents of a .diffs.<k> file.  Rows are split on '\t' exactly like make_bed.py:79-82 (8 fields, or 7
 * for the old format).  Loci come back in first-seen order (dict insertion order, :86-96, :134).
 * Returns number of loci, or <0 on malformed rows.
 */
int64_t orc_aggregate(const char *text, int64_t nbytes, orc_locus *loci, int64_t cap)
{
    int64_t n = 0;
    int64_t tsz = 1; while (tsz < 2 * cap + 16) tsz <<= 1;
    int64_t *table = (int64_t *)malloc(sizeof(int64_t) * (size_t)tsz);
    for (int64_t i = 0; i < tsz; i++) table[i] = -1;
    const char *p = text, *end = text + nbytes;
    int64_t rc = 0;
    while (p < end) {
        const char *nl = (const char *)memchr(p, '\n', (size_t)(end - p));
        const char *le = nl ? nl + 1 : end;      /* python keeps the '\n' inside the last field */
        tok_t f[9]; int nf = 0; const char *s = p;
        for (const char *q = p; q <= le; q++) {
            if (q == le || *q == '\t') { if (nf < 9) { f[nf].p = s; f[nf].len = (int)(q - s); } nf++; s = q + 1; }
        }
        p = le;
        if (nf != 8 && nf != 7) { rc = -1; goto done; }
        tok_t csome = f[0], pos = f[2], context = f[3], strand = f[5], label = f[6];
        int64_t posv; if (parse_i64(pos, &posv)) { rc = -1; goto done; }
        if (context.len == 0 || context.p[context.len / 2] != 'M') continue;     /* :84 */
        uint64_t h = fnv(csome.p, csome.len, 1469598103934665603ULL);
        h = fnv("\t", 1, h); h = fnv(pos.p, pos.len, h); h = fnv("\t", 1, h);
        h = fnv(context.p, context.len, h); h = fnv("\t", 1, h); h = fnv(strand.p, strand.len, h);
        int64_t slot = (int64_t)(h & (uint64_t)(tsz - 1));
        int64_t idx = -1;
        while (table[slot] >= 0) {
            orc_locus *L = &loci[table[slot]];
            tok_t k0 = { text + L->key_off[0], L->key_len[0] }, k1 = { text + L->key_off[1], L->key_len[1] },
                  k2 = { text + L->key_off[2], L->key_len[2] }, k3 = { text + L->key_off[3], L->key_len[3] };
            if (tok_eq(k0, csome) && tok_eq(k1, pos) && tok_eq(k2, context) && tok_eq(k3, strand)) { idx = table[slot]; break; }
            slot = (slot + 1) & (tsz - 1);
        }
        if (idx < 0) {
            if (n >= cap) { rc = ERR_CAP; goto done; }
            idx = n++;
            table[slot] = idx;
            orc_locus *L = &loci[idx];
            memset(L, 0, sizeof(*L));
            L->key_off[0] = csome.p - text; L->key_len[0] = csome.len;
            L->key_off[1] = pos.p - text; L->key_len[1] = pos.len;
            L->key_off[2] = context.p - text; L->key_len[2] = context.len;
            L->key_off[3] = strand.p - text; L->key_len[3] = strand.len;
        }
        loci[idx].depth++;
        if (label.len > 0 && label.p[0] == 'm') loci[idx].meth++;                /* :93-96 */
    }
    rc = n;
done:
    free(table);
    return rc;
}

int32_t orc_sizeof_locus(void) { return (int32_t)sizeof(orc_locus); }
