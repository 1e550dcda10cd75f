/* TEST INFRASTRUCTURE ONLY -- never linked into, imported by, or called from the
 * product path (navtex_b200/).  Only tests/, __graft_entry__.smoke() and
 * bench.py's cpu_baseline / --impl reference legs may use it.
 *
 * navtex_oracle: a plain-C, FP64, one-sample-at-a-time restatement of the
 * reference receive chain
 *     fir1cpp -> NCO mix -> fir2cpp -> fir3cpp -> decoder -> nav_b_sm
 * (reference files under /root/reference/receiver/, cited per function in the
 * .c file).  It exists for what the unmodified reference cannot express:
 * per-channel NCO offsets other than +-14 kHz and alternative tap sets, and as a
 * portable checker on the GPU box.
 *
 * PARITY PINNING: the reference ships no tests / golden vectors (SURVEY.md 4,
 * 8c).  This restatement is pinned by EXECUTION: tests/test_oracle.py
 * runs the unmodified reference (oracle/_ref/ref_chain) and this library on the
 * same inputs and requires exact FP64 equality of every stage tap, exact bit
 * strings and exact messages; tests/golden/ holds fixtures generated from
 * oracle/_ref/ref_chain (generator script committed beside them) so the same
 * check runs where /root/reference does not exist.
 */
#ifndef NAVTEX_ORACLE_H
#define NAVTEX_ORACLE_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct nvo_chain nvo_chain;
#define NVO_MAX_CH 8

typedef struct {
    /* NULL taps = the reference's literal arrays (fir1cpp.C:10-49, fir2cpp.C:24-72, fir3cpp.h:17-89) */
    const double *h1; int n1;
    const double *h2; int n2;
    const double *h3; int n3;
    /* channel NCO shifts in Hz at the 63 kHz rate; reference = +14000 ("518"), -14000 ("490").  Channels beyond the
     * reference's two (n_channels > 2: more channels of one capture sharing stage 1, SURVEY.md 8f.4) repeat the per-channel
     * half of fir2cpp.C:112-215 / nav_sched.C:10-16 with their own offset */
    double nco_hz[NVO_MAX_CH];
    /* table period in 63 kHz samples; 0 = derive (9 for +-14 kHz, fir2cpp.C:12-14) */
    int nco_period[NVO_MAX_CH];
    int freq_tag[NVO_MAX_CH]; /* passed through to messages; reference 518 / 490 */
    int record_taps;          /* keep y1/y2/y3 arrays (memory!) */
    int n_channels;           /* 0 = 2 (the reference) */
} nvo_params;

void nvo_default_params(nvo_params *p);
nvo_chain *nvo_new(const nvo_params *p);        /* NULL = reference defaults */
void nvo_free(nvo_chain *c);

/* feed n IQ samples (interleaved I,Q doubles), exactly like n calls of sample_in_1 */
void nvo_push(nvo_chain *c, const double *iq, size_t n);
void nvo_push_f32(nvo_chain *c, const float *iq, size_t n);
void nvo_push_s16(nvo_chain *c, const int16_t *iq, size_t n);
/* feed n 900 Hz samples (interleaved I,Q doubles) straight to channel ch's decoder and state machine, as if they had come out of
 * its third filter stage; y3 records them.  For tests of the demodulator alone.  A chain is fed through nvo_push* or through
 * nvo_push_900, never both: the 900 Hz sample counts (bitpos, pick margins) would no longer match either input */
void nvo_push_900(nvo_chain *c, int ch, const double *iq, size_t n);

/* recorded taps; pointers stay valid until the next push.  counts are complex samples */
size_t nvo_y1(const nvo_chain *c, const double **iq);
size_t nvo_y2(const nvo_chain *c, int ch, const double **iq);
size_t nvo_y3(const nvo_chain *c, int ch, const double **iq);
size_t nvo_bits(const nvo_chain *c, int ch, const char **bits);          /* 'B' / 'Y' */
size_t nvo_bitpos(const nvo_chain *c, int ch, const int32_t **pos);      /* 900 Hz sample count at decision */
/* per bit-sync evaluation (decoder.C:204-215): pairs (900 Hz sample count, (best - runner-up) / best of the nine sums) */
size_t nvo_pick_margins(const nvo_chain *c, int ch, const double **pairs);
size_t nvo_disc(const nvo_chain *c, int ch, const float **sums);         /* 4 floats per bit: BR BI YR YI */
/* every character appended to a line, '\n' for a completed line, 0x18 for an abort (in order) */
size_t nvo_events(const nvo_chain *c, int ch, const char **ev);

size_t nvo_n_messages(const nvo_chain *c);
/* message k in add_message call order */
int nvo_message(const nvo_chain *c, size_t k, int *freq, const char **bbbb, const char **text);

/* stand-alone pieces, for unit tests of the CUDA kernels */
typedef struct nvo_decoder nvo_decoder;
nvo_decoder *nvo_decoder_new(void);
void nvo_decoder_free(nvo_decoder *d);
/* returns 'B'/'Y' when this 900 Hz sample completed a bit, else 0; sums (4 floats) optional */
char nvo_decoder_sample(nvo_decoder *d, double i, double q, float *sums);

#ifdef __cplusplus
}
#endif
#endif
