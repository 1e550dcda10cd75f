/* TEST INFRASTRUCTURE ONLY -- see navtex_oracle.h.
 *
 * Plain-C FP64 restatement of the reference receive chain, one sample per
 * call, same operation order as the reference so that results are bit-equal
 * to the compiled reference at the default parameters (checked by
 * tests/test_oracle.py).  Build with -ffp-contract=off and no -march
 * so that, like the reference build (-O3 only, receiver/configure.ac:3-4),
 * no multiply-add is fused.
 *
 * All "ref:" citations are relative to /root/reference/receiver/.
 */
#define _GNU_SOURCE
#include "navtex_oracle.h"
#include "../include/navtex_taps.h"

#include <math.h>
#include <regex.h>
#include <stdlib.h>
#include <string.h>

static const double k_h1[NVX_T1] = {NVX_H1_VALUES};
static const double k_h2[NVX_T2] = {NVX_H2_VALUES};
static const double k_h3[NVX_T3] = {NVX_H3_VALUES};

/* ------------------------------------------------------------------ utils */
typedef struct { char *p; size_t n, cap; } bytes_t;
static void bytes_add(bytes_t *b, const void *src, size_t n) {
    if (b->n + n > b->cap) {
        size_t cap = b->cap ? b->cap * 2 : 4096;
        while (cap < b->n + n) cap *= 2;
        b->p = (char *)realloc(b->p, cap);
        b->cap = cap;
    }
    memcpy(b->p + b->n, src, n);
    b->n += n;
}
static void bytes_add_c(bytes_t *b, char c) { bytes_add(b, &c, 1); }
static void bytes_add_2d(bytes_t *b, double x, double y) { double v[2] = {x, y}; bytes_add(b, v, sizeof v); }

/* ------------------------------------------------------- decimating FIR
 * One algorithm, three instances (SURVEY.md A.1):
 *   ref: fir1cpp.C:80-136 (T=37, D=4, ring 4096, AoS)
 *   ref: fir2cpp.C:131-171 and :175-215 (T=47, D=7, ring 1024, SoA)
 *   ref: fir3cpp.C:22-60 (T=71, D=10, ring 1024)
 * store at ptr; ++count; on count%D==0 sum h[0]*newest ... h[T-1]*oldest in
 * that order, emit, count=0; ptr=(ptr+1)%L.  The ring length has no numerical
 * effect as long as L >= T (fir1cpp.C:101 is only a no-wrap fast path).       */
typedef struct {
    const double *h;
    int T, D, L;
    double *ri, *rq;
    int ptr, count;
} fir_t;

static void fir_init(fir_t *f, const double *h, int T, int D, int min_ring) {
    int L = min_ring;
    while (L < T + 1) L *= 2;
    f->h = h; f->T = T; f->D = D; f->L = L;
    f->ri = (double *)calloc((size_t)L, sizeof(double));   /* zero history: fir1cpp.C:72-76, fir2cpp.C:96-100, fir3cpp.C:12-16 */
    f->rq = (double *)calloc((size_t)L, sizeof(double));
    f->ptr = 0; f->count = 0;
}
static void fir_free(fir_t *f) { free(f->ri); free(f->rq); }

static int fir_push(fir_t *f, double xi, double xq, double *yi, double *yq) {
    int fired = 0;
    f->ri[f->ptr] = xi;
    f->rq[f->ptr] = xq;
    f->count++;
    if (f->count % f->D == 0) {
        double si = 0.0, sq = 0.0;
        int at = f->ptr;
        for (int t = 0; t < f->T; ++t) {
            double c = f->h[t];
            si += c * f->ri[at];
            sq += c * f->rq[at];
            at = at == 0 ? f->L - 1 : at - 1;
        }
        *yi = si; *yq = sq;
        f->count = 0;
        fired = 1;
    }
    f->ptr = (f->ptr + 1) % f->L;
    return fired;
}

/* ------------------------------------------------------------------ NCO
 * ref: fir2cpp.C:104-107 (table), :112-128 (mix).  Table entry i is
 * (cos(x), -sin(x)), x = (2*M_PI*i*F)/FS evaluated left to right in double;
 * the index advances once per 63 kHz sample and wraps at the table period.
 * Channel "518" multiplies by (re + j im); channel "490" uses the conjugate,
 * which is the same formula with F = -14000 (cos even, sin odd: bit-equal). */
typedef struct { double *re, *im; int period, at; } nco_t;

static int nco_period_for(double f_hz) {
    /* smallest P with P*f/63000 integer, f on a 0.5 Hz grid */
    long num = lround(fabs(f_hz) * 2.0), den = 126000;
    if (num == 0) return 1;
    long a = num, b = den;
    while (b) { long t = a % b; a = b; b = t; }
    return (int)(den / a);
}
static void nco_init(nco_t *n, double f_hz, int period) {
    if (period <= 0) period = nco_period_for(f_hz);
    n->period = period; n->at = 0;
    n->re = (double *)malloc(sizeof(double) * (size_t)period);
    n->im = (double *)malloc(sizeof(double) * (size_t)period);
    for (int i = 0; i < period; ++i) {
        n->re[i] = cos((2 * M_PI * i * f_hz) / 63000);
        n->im[i] = -sin((2 * M_PI * i * f_hz) / 63000);
    }
}
static void nco_free(nco_t *n) { free(n->re); free(n->im); }

/* ---------------------------------------------------------------- decoder */
enum { DS_INIT = 0, DS_WAIT = 1, DS_BIT_START = 2, DS_RECEIVING = 3 };   /* ref: decoder.h:16-19 */
#define SPB 9            /* samples per bit, decoder.h:21 */
#define CORR_LEN (63 * SPB) /* decoder.h:23-24 */
#define N_BURN 2         /* decoder.h:10 */
#define N_USE 5          /* decoder.h:11 */

struct nvo_decoder {
    double prev_i, prev_q;
    /* timing recovery */
    double ang[SPB];  int ang_at, ang_full;
    double corr[CORR_LEN]; int corr_at, corr_full;
    double osum[SPB]; int osum_at, osum_full;
    int sync_tick;          /* bs_seq_nbr */
    int last_pick;          /* prev_offset */
    /* not in the reference: how close the last arg max was, (best - runner-up) / best, for the parity reports of the tests
     * (a GPU / CPU difference in the last bits of the sums can only flip a pick at a near-tie) */
    double pick_margin; int pick_fresh;
    /* mark/space discriminator */
    int state, tick, offs, next_offs, burned, used;
    float br, bi, yr, yi;
    float tone_r[N_USE], tone_i[N_USE];
};

/* ref: decoder.C:6-39 */
static void decoder_init(nvo_decoder *d) {
    memset(d, 0, sizeof *d);
    d->state = DS_INIT;
    d->last_pick = -1;
    for (int i = 0; i < N_USE; ++i) {
        float a = (float)((i * 2 * 3.1415 * 85) / 900);      /* 3.1415, not pi: decoder.C:25 */
        d->tone_r[i] = cosf(a);                               /* C++ cos(float) is the float overload */
        d->tone_i[i] = sinf(a);
    }
}

/* ref: decoder.C:62-70 */
static void decoder_set_sync(nvo_decoder *d, int offs) {
    if (d->state == DS_INIT) { d->state = DS_WAIT; d->offs = offs; }
    d->next_offs = offs;
}

/* ref: decoder.C:142-255 */
static void decoder_timing(nvo_decoder *d, double angle) {
    static const int mask[SPB] = {0, 1, 1, 1, 0, -1, -1, -1, 0};   /* decoder.h:62-72 */
    d->ang[d->ang_at] = angle;
    if (++d->ang_at == SPB) { d->ang_at = 0; d->ang_full = 1; }
    if (d->ang_full) {
        double acc = 0.0;
        int j = d->ang_at;                     /* oldest first */
        for (int i = 0; i < SPB; ++i) {
            acc += mask[i] * d->ang[j];
            j = (j + 1) % SPB;
        }
        d->corr[d->corr_at] = fabs(acc);
        if (++d->corr_at == CORR_LEN) { d->corr_at = 0; d->corr_full = 1; }
    }
    if (d->corr_full) {
        double acc = 0.0;
        for (int i = d->osum_at; i < CORR_LEN; i += SPB) acc += d->corr[i];   /* ascending ring index */
        d->osum[d->osum_at] = acc;
        if (++d->osum_at == SPB) { d->osum_at = 0; d->osum_full = 1; }
    }
    if (d->osum_full) {
        if (d->sync_tick % SPB == 0) {
            double best = -1.0;
            int pick = 0;
            for (int i = 0; i < SPB; ++i)
                if (d->osum[i] > best) { best = d->osum[i]; pick = i; }
            {
                double second = -1.0;
                for (int i = 0; i < SPB; ++i)
                    if (i != pick && d->osum[i] > second) second = d->osum[i];
                d->pick_margin = best > 0.0 ? (best - second) / best : 0.0;
                d->pick_fresh = 1;
            }
            if (d->last_pick != -1 && pick != d->last_pick) {
                /* slew by exactly one step toward the new maximum, the short way round (decoder.C:217-246) */
                int up;
                if (pick > d->last_pick) up = !(pick - d->last_pick > 4);
                else up = (d->last_pick - pick > 4);
                pick = up ? (d->last_pick + 1) % SPB : (d->last_pick - 1 + SPB) % SPB;
            }
            d->last_pick = pick;
            decoder_set_sync(d, (pick + 5) % SPB);
        }
        d->sync_tick = (d->sync_tick + 1) % SPB;
    }
}

/* ref: decoder.C:73-137; accumulator arithmetic per SURVEY.md A.3 (cast binds
 * tighter than '*': first product in float, second in double, sum in double,
 * stored back to float). */
static char decoder_discriminate(nvo_decoder *d, double s_r, double s_i) {
    d->tick++;
    if (d->state == DS_INIT) return 0;
    if (d->state == DS_WAIT && d->tick % SPB == d->offs) { d->state = DS_BIT_START; d->burned = 0; }
    if (d->state == DS_BIT_START) {
        if (d->burned == N_BURN) {
            d->state = DS_RECEIVING; d->used = 0;
            d->br = d->bi = d->yr = d->yi = 0.0f;
        } else {
            d->burned++;
        }
        return 0;
    }
    if (d->state == DS_RECEIVING) {
        const float fr = d->tone_r[d->used], fi = d->tone_i[d->used];
        const float sr_f = (float)s_r, nsr_f = (float)-s_r;
        d->yr = (float)((double)d->yr + ((double)(sr_f * fr) - s_i * (double)fi));
        d->yi = (float)((double)d->yi + ((double)(sr_f * fi) + s_i * (double)fr));
        d->br = (float)((double)d->br + ((double)(sr_f * fr) + s_i * (double)fi));
        d->bi = (float)((double)d->bi + ((double)(nsr_f * fi) + s_i * (double)fr));
        if (++d->used == N_USE) {
            float p1 = d->br * d->br, p2 = d->bi * d->bi;
            float q1 = d->yr * d->yr, q2 = d->yi * d->yi;
            float eb = p1 + p2, ey = q1 + q2;
            d->state = DS_WAIT;
            d->offs = d->next_offs;
            return eb > ey ? 'B' : 'Y';
        }
    }
    return 0;
}

/* ref: decoder.C:42-59 */
char nvo_decoder_sample(nvo_decoder *d, double i, double q, float *sums) {
    double re = i * d->prev_i + q * d->prev_q;
    double im = q * d->prev_i - i * d->prev_q;
    double angle = atan2(im, re);
    d->prev_i = i; d->prev_q = q;
    decoder_timing(d, angle);
    char bit = decoder_discriminate(d, i, q);
    if (bit && sums) { sums[0] = d->br; sums[1] = d->bi; sums[2] = d->yr; sums[3] = d->yi; }
    return bit;
}
nvo_decoder *nvo_decoder_new(void) {
    nvo_decoder *d = (nvo_decoder *)malloc(sizeof *d);
    decoder_init(d);
    return d;
}
void nvo_decoder_free(nvo_decoder *d) { free(d); }

/* ------------------------------------------------- SITOR-B / CCIR 476 FSM
 * ref: nav_b_sm.h:60-83 (tables), nav_b_sm.C.  The table is written here as
 * (code, letters-case, figures-case) triples; every code not listed is
 * invalid ('_').  Lower-case marks are controls: p = alpha (phasing 1),
 * q = RQ (phasing 2), l = LTRS, f = FIGS, n = LF, r = CR.  0x5c decodes as a
 * space although it is not a 3-of-7 code, and 0x1d has a figures entry but no
 * letters entry (so it is invalid): both are kept, they are results. */
static const struct { unsigned char code; char l, f; } k_codes[] = {
    {0x07, 'p', 'p'}, {0x0b, 'J', 'b'}, {0x0d, 'W', '2'}, {0x0e, 'A', '-'}, {0x13, 'F', '*'},
    {0x15, 'Y', '6'}, {0x16, 'S', '\''}, {0x19, '-', '-'}, {0x1a, 'D', '%'}, {0x1c, 'Z', '+'},
    {0x1d, '_', ' '}, {0x23, 'C', ':'}, {0x25, 'P', '0'}, {0x26, 'I', '8'}, {0x29, 'G', '*'},
    {0x2a, 'R', '4'}, {0x2c, 'L', ')'}, {0x31, 'M', '.'}, {0x32, 'N', ','}, {0x34, 'H', '*'},
    {0x38, 'O', '9'}, {0x43, 'K', '('}, {0x45, 'Q', '1'}, {0x46, 'U', '7'}, {0x49, 'f', 'f'},
    {0x4a, 'E', '3'}, {0x4c, 'q', 'q'}, {0x51, 'X', '/'}, {0x52, 'l', 'l'}, {0x58, 'B', '?'},
    {0x5c, ' ', ' '}, {0x61, 'V', '='}, {0x62, ' ', ' '}, {0x64, 'n', 'n'}, {0x68, 'T', '5'},
    {0x70, 'r', 'r'},
};
static unsigned char g_ltrs[128], g_figs[128];
static int g_tables_ready;
static void tables_init(void) {
    if (g_tables_ready) return;
    memset(g_ltrs, '_', sizeof g_ltrs);
    memset(g_figs, '_', sizeof g_figs);
    for (size_t k = 0; k < sizeof k_codes / sizeof k_codes[0]; ++k) {
        g_ltrs[k_codes[k].code] = (unsigned char)k_codes[k].l;
        g_figs[k_codes[k].code] = (unsigned char)k_codes[k].f;
    }
    g_tables_ready = 1;
}

#define CODE_ALPHA 0x07   /* ph1, nav_b_sm.h:89 */
#define CODE_RQ 0x4c      /* ph2, nav_b_sm.h:90 */
#define ERR_WINDOW 20     /* nav_b_sm.h:49 */
#define ERR_LIMIT 12      /* nav_b_sm.h:50 */
#define HOLDOFF_BITS 1100 /* nav_b_sm.h:52 */
#define TEXT_CAP 5000     /* nav_b_sm.h:97-98 */
#define EV_ABORT 0x18

/* the 30-bit phasing pattern walked by nav_b_sm.C:296-630: ...RQ alpha RQ alpha RQ */
static const char k_phasing[] = "BBBBBBYYYYBBYYBBBBBBYYYYBBYYBB";

enum { BY_WAIT = 1, BY_GOT_DX = 2, BY_GOT_RX = 3 };   /* nav_b_sm.h:41-43 */

typedef struct { int freq; char bbbb[10]; char *text; } msg_t;

typedef struct nvo_bsm {
    int freq;
    int match;                 /* status: bits of k_phasing matched so far */
    int byte_state, figures;
    int nbits; char shift;     /* bits_received, temp_byte */
    char dx_ring[3]; int dx_at, dx_full;
    char err_ring[ERR_WINDOW]; int err_at, err_full, err_count;
    int eoe_count, prev_dx_alpha;
    int holdoff;
    int enabled, in_message;
    char line[TEXT_CAP], text[TEXT_CAP], bbbb[10];
    regex_t re_som, re_eom;
    bytes_t events;
    struct nvo_chain *owner;
} nvo_bsm;

struct nvo_chain {
    nvo_params prm;
    int nch;
    fir_t f1, f2[NVO_MAX_CH], f3[NVO_MAX_CH];
    nco_t nco[NVO_MAX_CH];
    nvo_decoder dec[NVO_MAX_CH];
    nvo_bsm bsm[NVO_MAX_CH];
    long n3[NVO_MAX_CH];
    bytes_t y1, y2[NVO_MAX_CH], y3[NVO_MAX_CH], bits[NVO_MAX_CH], bitpos[NVO_MAX_CH], disc[NVO_MAX_CH], pickm[NVO_MAX_CH];
    msg_t *msgs; size_t n_msgs, cap_msgs;
};

static void chain_add_message(struct nvo_chain *c, const char *bbbb, const char *text, int freq) {
    if (c->n_msgs == c->cap_msgs) {
        c->cap_msgs = c->cap_msgs ? c->cap_msgs * 2 : 8;
        c->msgs = (msg_t *)realloc(c->msgs, c->cap_msgs * sizeof(msg_t));
    }
    msg_t *m = &c->msgs[c->n_msgs++];
    m->freq = freq;
    strncpy(m->bbbb, bbbb, sizeof m->bbbb - 1);
    m->bbbb[sizeof m->bbbb - 1] = 0;
    m->text = strdup(text);
}

/* bounded append (the reference strcat()s without bounds into 5000-byte buffers,
 * nav_b_sm.h:97-98; overflowing them is undefined there, clamped here) */
static void text_append(char *dst, const char *src, size_t n) {
    size_t have = strlen(dst);
    if (have + n > TEXT_CAP - 1) n = TEXT_CAP - 1 - have;
    memcpy(dst + have, src, n);
    dst[have + n] = 0;
}

/* ref: nav_b_sm.C:16-42 */
static void bsm_reset(nvo_bsm *s) {
    s->match = 0;
    s->byte_state = BY_WAIT;
    s->figures = 0;
    s->nbits = 0;
    s->dx_at = 0; s->dx_full = 0;
    s->err_count = 0; s->err_at = 0; s->err_full = 0;   /* ring contents are NOT cleared */
    s->eoe_count = 0; s->prev_dx_alpha = 0;
    s->line[0] = 0; s->text[0] = 0; s->bbbb[0] = 0;
    s->holdoff = 0;
    s->enabled = 0; s->in_message = 0;
}

/* ref: nav_b_sm.C:44-52 */
static void bsm_abort(nvo_bsm *s) {
    bytes_add_c(&s->events, EV_ABORT);
    if (s->in_message) chain_add_message(s->owner, s->bbbb, s->text, s->freq);
    bsm_reset(s);
}

/* ref: nav_b_sm.C:56-97 */
static void bsm_line_done(nvo_bsm *s) {
    regmatch_t m[4];
    bytes_add_c(&s->events, '\n');
    if (s->in_message) {
        text_append(s->text, s->line, strlen(s->line));
        text_append(s->text, "\n", 1);
    }
    if (regexec(&s->re_som, s->line, 4, m, 0) == 0) {
        s->text[0] = 0;
        text_append(s->text, s->line, strlen(s->line));
        text_append(s->text, "\n", 1);
        /* strncat onto whatever bbbb already holds, then cut at 4 (nav_b_sm.C:74-76) */
        size_t have = strlen(s->bbbb);
        size_t n2 = (size_t)(m[2].rm_eo - m[2].rm_so), n3 = (size_t)(m[3].rm_eo - m[3].rm_so);
        if (have + n2 + n3 < sizeof s->bbbb) {
            memcpy(s->bbbb + have, s->line + m[2].rm_so, n2);
            memcpy(s->bbbb + have + n2, s->line + m[3].rm_so, n3);
            s->bbbb[have + n2 + n3] = 0;
        }
        s->bbbb[4] = 0;
        s->in_message = 1;
    } else if (regexec(&s->re_eom, s->line, 1, m, 0) == 0) {
        if (s->in_message) chain_add_message(s->owner, s->bbbb, s->text, s->freq);
        s->text[0] = 0;
        s->bbbb[0] = 0;
        s->in_message = 0;
    }
    s->line[0] = 0;
}

/* ref: nav_b_sm.C:100-145 */
static void bsm_char_out(nvo_bsm *s, unsigned char code) {
    char out;
    if (code == 0) out = '*';
    else {
        unsigned char l = g_ltrs[code];
        if (l == 'l') { s->figures = 0; return; }
        if (l == 'f') { s->figures = 1; return; }
        if (l == 'n') { bsm_line_done(s); return; }
        if (l == 'r' || l == 'p' || l == 'q') return;
        out = (char)(s->figures ? g_figs[code] : l);
    }
    bytes_add_c(&s->events, out);
    text_append(s->line, &out, 1);
}

/* ref: nav_b_sm.C:150-262 */
static void bsm_byte(nvo_bsm *s, unsigned char b) {
    switch (s->byte_state) {
    case BY_WAIT:
        if (b == CODE_ALPHA) s->byte_state = BY_GOT_RX;
        if (b == CODE_RQ) s->byte_state = BY_GOT_DX;
        break;
    case BY_GOT_RX: {        /* this byte sits in the DX slot */
        int stop = 0;
        s->dx_ring[s->dx_at] = (char)b;
        if (++s->dx_at == 3) { s->dx_at = 0; s->dx_full = 1; }
        if (b == CODE_ALPHA) {
            if (s->prev_dx_alpha && ++s->eoe_count == 2) { bsm_abort(s); stop = 1; }   /* end of emission */
            if (!stop) s->prev_dx_alpha = 1;
        } else {
            s->prev_dx_alpha = 0;
        }
        if (!stop) s->byte_state = BY_GOT_DX;
        break;
    }
    case BY_GOT_DX:          /* this byte sits in the RX slot */
        if (s->dx_full) {
            unsigned char dx = (unsigned char)s->dx_ring[s->dx_at];
            if (g_ltrs[b] != '_') bsm_char_out(s, b);
            else if (g_ltrs[dx & 0x7f] != '_') bsm_char_out(s, dx);
            else bsm_char_out(s, 0);
        }
        s->byte_state = BY_GOT_RX;
        break;
    }
    /* sliding window of invalid codes over every byte, phasing included (nav_b_sm.C:235-261) */
    if (s->err_full && s->err_ring[s->err_at] == '_') s->err_count--;
    s->err_ring[s->err_at] = (char)g_ltrs[b];
    if (s->err_ring[s->err_at] == '_') s->err_count++;
    if (++s->err_at == ERR_WINDOW) { s->err_at = 0; s->err_full = 1; }
    if (s->err_count > ERR_LIMIT) {
        bsm_char_out(s, 0);
        bsm_abort(s);
    }
}

/* ref: nav_b_sm.C:266-634 */
static void bsm_bit(nvo_bsm *s, char bit) {
    if (s->enabled) {
        s->shift = (char)(s->shift << 1);
        if (bit == 'Y') s->shift |= 1;
        if (++s->nbits == 7) {
            bsm_byte(s, (unsigned char)s->shift & 0x7f);
            s->nbits = 0;
            s->shift = 0;
        }
    }
    if (s->holdoff != 0) { s->holdoff--; return; }
    if (s->match == 29) {                   /* last state: any bit returns to INIT (nav_b_sm.C:618-630) */
        if (bit == 'B') {
            s->enabled = 1; s->nbits = 0; s->shift = 0;
            s->holdoff = HOLDOFF_BITS;
        }
        s->match = 0;
    } else if (bit == k_phasing[s->match]) {
        s->match++;
    } else if (s->match == 6) {
        /* only the first run of B's tolerates extra B's (nav_b_sm.C:363-372) */
    } else {
        s->match = 0;                       /* not re-seeded with the current bit */
    }
}

static void bsm_init(nvo_bsm *s, struct nvo_chain *owner, int freq) {
    memset(s, 0, sizeof *s);
    s->owner = owner; s->freq = freq;
    regcomp(&s->re_som, "(CZC|Z.ZC|ZC.C|ZCZ.) +([A-Z][A-Z])([0-9][0-9])", REG_EXTENDED);   /* nav_b_sm.C:69 */
    regcomp(&s->re_eom, "NNN.*|N.NN.*|NN.N.*", REG_EXTENDED);                               /* nav_b_sm.C:80 */
    bsm_reset(s);
}

/* ------------------------------------------------------------------ chain */
void nvo_default_params(nvo_params *p) {
    memset(p, 0, sizeof *p);
    p->nco_hz[0] = 14000.0; p->nco_hz[1] = -14000.0;
    p->freq_tag[0] = 518; p->freq_tag[1] = 490;      /* nav_sched.C:10-11 */
    p->record_taps = 1;
}

nvo_chain *nvo_new(const nvo_params *prm) {
    tables_init();
    nvo_chain *c = (nvo_chain *)calloc(1, sizeof *c);
    if (prm) c->prm = *prm; else nvo_default_params(&c->prm);
    const nvo_params *p = &c->prm;
    c->nch = p->n_channels > 0 && p->n_channels <= NVO_MAX_CH ? p->n_channels : 2;
    fir_init(&c->f1, p->h1 ? p->h1 : k_h1, p->h1 ? p->n1 : NVX_T1, NVX_D1, 4096);
    for (int ch = 0; ch < c->nch; ++ch) {
        fir_init(&c->f2[ch], p->h2 ? p->h2 : k_h2, p->h2 ? p->n2 : NVX_T2, NVX_D2, 1024);
        fir_init(&c->f3[ch], p->h3 ? p->h3 : k_h3, p->h3 ? p->n3 : NVX_T3, NVX_D3, 1024);
        nco_init(&c->nco[ch], p->nco_hz[ch], p->nco_period[ch]);
        decoder_init(&c->dec[ch]);
        bsm_init(&c->bsm[ch], c, p->freq_tag[ch]);
    }
    return c;
}

void nvo_free(nvo_chain *c) {
    if (!c) return;
    fir_free(&c->f1);
    for (int ch = 0; ch < c->nch; ++ch) {
        fir_free(&c->f2[ch]); fir_free(&c->f3[ch]); nco_free(&c->nco[ch]);
        regfree(&c->bsm[ch].re_som); regfree(&c->bsm[ch].re_eom);
        free(c->bsm[ch].events.p);
        free(c->y2[ch].p); free(c->y3[ch].p); free(c->bits[ch].p); free(c->bitpos[ch].p); free(c->disc[ch].p); free(c->pickm[ch].p);
    }
    free(c->y1.p);
    for (size_t k = 0; k < c->n_msgs; ++k) free(c->msgs[k].text);
    free(c->msgs);
    free(c);
}

/* the per-channel tail of the chain: one 900 Hz sample into channel ch's decoder and state machine, with its taps recorded */
static void chain_900(nvo_chain *c, int ch, double ci, double cq) {
    if (c->prm.record_taps) bytes_add_2d(&c->y3[ch], ci, cq);
    c->n3[ch]++;
    float sums[4];
    char bit = nvo_decoder_sample(&c->dec[ch], ci, cq, sums);
    if (c->dec[ch].pick_fresh) {
        c->dec[ch].pick_fresh = 0;
        if (c->prm.record_taps) { double rec[2] = {(double)c->n3[ch], c->dec[ch].pick_margin}; bytes_add(&c->pickm[ch], rec, sizeof rec); }
    }
    if (bit) {
        int32_t pos = (int32_t)c->n3[ch];
        bytes_add_c(&c->bits[ch], bit);
        bytes_add(&c->bitpos[ch], &pos, sizeof pos);
        bytes_add(&c->disc[ch], sums, sizeof sums);
        bsm_bit(&c->bsm[ch], bit);
    }
}

static void chain_sample(nvo_chain *c, double xi, double xq) {
    double ai, aq;
    if (!fir_push(&c->f1, xi, xq, &ai, &aq)) return;
    if (c->prm.record_taps) bytes_add_2d(&c->y1, ai, aq);
    for (int ch = 0; ch < c->nch; ++ch) {
        /* ref: fir2cpp.C:115-124 */
        nco_t *n = &c->nco[ch];
        double re = n->re[n->at], im = n->im[n->at];
        double mi = ai * re - aq * im;
        double mq = ai * im + aq * re;
        n->at = (n->at + 1) % n->period;
        double bi, bq, ci, cq;
        if (!fir_push(&c->f2[ch], mi, mq, &bi, &bq)) continue;
        if (c->prm.record_taps) bytes_add_2d(&c->y2[ch], bi, bq);
        if (!fir_push(&c->f3[ch], bi, bq, &ci, &cq)) continue;
        chain_900(c, ch, ci, cq);
    }
}

void nvo_push(nvo_chain *c, const double *iq, size_t n) {
    for (size_t k = 0; k < n; ++k) chain_sample(c, iq[2 * k], iq[2 * k + 1]);
}
void nvo_push_f32(nvo_chain *c, const float *iq, size_t n) {
    for (size_t k = 0; k < n; ++k) chain_sample(c, (double)iq[2 * k], (double)iq[2 * k + 1]);
}
void nvo_push_s16(nvo_chain *c, const int16_t *iq, size_t n) {
    for (size_t k = 0; k < n; ++k) chain_sample(c, (double)iq[2 * k], (double)iq[2 * k + 1]);   /* capt_sched.c:511 */
}
void nvo_push_900(nvo_chain *c, int ch, const double *iq, size_t n) {
    if (ch < 0 || ch >= c->nch) return;
    for (size_t k = 0; k < n; ++k) chain_900(c, ch, iq[2 * k], iq[2 * k + 1]);
}

size_t nvo_y1(const nvo_chain *c, const double **iq) { *iq = (const double *)c->y1.p; return c->y1.n / 16; }
size_t nvo_y2(const nvo_chain *c, int ch, const double **iq) { *iq = (const double *)c->y2[ch].p; return c->y2[ch].n / 16; }
size_t nvo_y3(const nvo_chain *c, int ch, const double **iq) { *iq = (const double *)c->y3[ch].p; return c->y3[ch].n / 16; }
size_t nvo_bits(const nvo_chain *c, int ch, const char **b) { *b = c->bits[ch].p; return c->bits[ch].n; }
size_t nvo_bitpos(const nvo_chain *c, int ch, const int32_t **p) { *p = (const int32_t *)c->bitpos[ch].p; return c->bitpos[ch].n / 4; }
size_t nvo_disc(const nvo_chain *c, int ch, const float **s) { *s = (const float *)c->disc[ch].p; return c->disc[ch].n / 16; }
size_t nvo_pick_margins(const nvo_chain *c, int ch, const double **m) { *m = (const double *)c->pickm[ch].p; return c->pickm[ch].n / 16; }
size_t nvo_events(const nvo_chain *c, int ch, const char **e) { *e = c->bsm[ch].events.p; return c->bsm[ch].events.n; }
size_t nvo_n_messages(const nvo_chain *c) { return c->n_msgs; }
int nvo_message(const nvo_chain *c, size_t k, int *freq, const char **bbbb, const char **text) {
    if (k >= c->n_msgs) return -1;
    *freq = c->msgs[k].freq; *bbbb = c->msgs[k].bbbb; *text = c->msgs[k].text;
    return 0;
}
