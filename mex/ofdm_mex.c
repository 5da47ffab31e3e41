/*
 * ofdm_mex.c -- MEX gateway: MATLAB / GNU Octave host code -> libofdm_b200 (C ABI, include/ofdm_b200.h).
 *
 *   out = ofdm_mex('OpName', arg1, arg2, ...)     OpName = the reference function's own name
 *
 * Build (on a host that has MATLAB or Octave -- neither exists in the authoring image, where this
 * file is compiled against mex/shim/mex.h and driven through ctypes by tests/test_gpu_mex.py):
 *   MATLAB:  mex -R2018a -I../include ofdm_mex.c -L../ofdm-course_b200/lib -lofdm_b200
 *   Octave:  mkoctfile --mex -I../include ofdm_mex.c -L../ofdm-course_b200/lib -lofdm_b200
 * R2018a interleaved complex (mxGetComplexDoubles) and legacy / Octave split complex
 * (mxGetPr/mxGetPi) are both handled.  The gateway only marshals: doubles -> the context's real
 * type, 0/1 double bits -> packed words, 1-based double indices -> int32, host <-> device copies.
 * No computation happens here and there is no CPU fallback: without an sm_100 GPU every op fails
 * with ofdm:ctx:nodevice.  The matlab/<Name>.m wrappers give each op the reference's signature.
 * The six sweep ops run on the device set of ofdm_mex('devices', ids) (0-based CUDA ids, default [0]: one context on
 * device 0); any other set runs them through one ofdm_group, every other op stays on device 0.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "mex.h"
#include "ofdm_b200.h"

#if defined(MX_HAS_INTERLEAVED_COMPLEX) && MX_HAS_INTERLEAVED_COMPLEX
#define OFDM_INTERLEAVED 1
#else
#define OFDM_INTERLEAVED 0
#endif

static ofdm_ctx* g_ctx = NULL;
static int g_prec = OFDM_PREC_F32;
/* the device set of the six sweep ops (ofdm_mex('devices', ids), 0-based CUDA ids): [0] runs them on g_ctx, any other set
 * on g_group, built on first use and rebuilt after a precision switch */
#define MAX_DEVICES 64
static int g_devices[MAX_DEVICES] = {0};
static int g_ndevices = 1;
static ofdm_group* g_group = NULL;

/* ---- scratch bookkeeping: everything allocated during one call is released on exit or error ---- */
#define MAX_TMP 96
static void* g_dev[MAX_TMP]; static int g_ndev = 0;
static void* g_host[MAX_TMP]; static int g_nhost = 0;
static void release_all(void) {
    int i;
    for (i = 0; i < g_ndev; ++i) ofdm_free(g_ctx, g_dev[i]);
    for (i = 0; i < g_nhost; ++i) free(g_host[i]);
    g_ndev = g_nhost = 0;
}
static void at_exit(void) {
    release_all();
    if (g_ctx) { ofdm_ctx_destroy(g_ctx); g_ctx = NULL; }
    ofdm_group_destroy(g_group); g_group = NULL;
}
static void fail(const char* id, const char* msg) { release_all(); mexErrMsgIdAndTxt(id, "%s", msg); }
static void fail_call(const char* op, const char* text) {
    char buf[640];
    strncpy(buf, op, 64); buf[64] = 0; strcat(buf, ": ");
    strncat(buf, text, 500);
    fail("ofdm:call:failed", buf);
}
static void chk(int rc, const char* op) { if (rc != OFDM_OK) fail_call(op, g_ctx ? ofdm_last_error(g_ctx) : "no context"); }
static void chk_group(int rc, const char* op) { if (rc != OFDM_OK) fail_call(op, ofdm_group_last_error(g_group)); }
static void* hostbuf(size_t bytes) {
    void* p = calloc(bytes ? bytes : 1, 1);
    if (!p || g_nhost >= MAX_TMP) fail("ofdm:mem:host", "host allocation failed");
    g_host[g_nhost++] = p;
    return p;
}
static void* devbuf(size_t bytes) {
    void* p = NULL;
    if (g_ndev >= MAX_TMP) fail("ofdm:mem:device", "too many device temporaries");
    chk(ofdm_malloc(g_ctx, &p, bytes), "ofdm_malloc");
    g_dev[g_ndev++] = p;
    return p;
}
static void ensure_ctx(void) {
    if (!g_ctx) {
        int rc = ofdm_ctx_create(&g_ctx, 0, g_prec);
        if (rc == OFDM_ERR_NODEVICE) mexErrMsgIdAndTxt("ofdm:ctx:nodevice", "no sm_100 GPU: ofdm_b200 has no CPU fallback");
        if (rc != OFDM_OK) mexErrMsgIdAndTxt("ofdm:ctx:create", "ofdm_ctx_create failed (%d)", rc);
        mexAtExit(at_exit);
    }
}
/* the group of the sweep ops, or NULL when the device set is the default [0] (the single-context path) */
static ofdm_group* sweep_group(void) {
    int rc;
    if (g_ndevices == 1 && g_devices[0] == 0) return NULL;
    if (g_group) return g_group;
    rc = ofdm_group_create(&g_group, g_devices, g_ndevices, g_prec);
    if (rc == OFDM_ERR_NODEVICE) fail("ofdm:devices:nodevice", "a device of the set is not an sm_100 GPU of this host");
    if (rc != OFDM_OK) mexErrMsgIdAndTxt("ofdm:devices:create", "ofdm_group_create failed (%d)", rc);
    return g_group;
}
static size_t esz(void) { return g_prec == OFDM_PREC_F64 ? 2 * sizeof(double) : 2 * sizeof(float); }
static size_t rsz(void) { return g_prec == OFDM_PREC_F64 ? sizeof(double) : sizeof(float); }

/* ---- marshalling ---- */
static void get_complex(const mxArray* a, size_t i, double* re, double* im) {
#if OFDM_INTERLEAVED
    if (mxIsComplex(a)) { mxComplexDouble* z = mxGetComplexDoubles(a); *re = z[i].real; *im = z[i].imag; }
    else { *re = mxGetDoubles(a)[i]; *im = 0.0; }
#else
    *re = mxGetPr(a)[i]; *im = mxIsComplex(a) ? mxGetPi(a)[i] : 0.0;
#endif
}
static void set_complex(mxArray* a, size_t i, double re, double im) {
#if OFDM_INTERLEAVED
    mxComplexDouble* z = mxGetComplexDoubles(a); z[i].real = re; z[i].imag = im;
#else
    mxGetPr(a)[i] = re; mxGetPi(a)[i] = im;
#endif
}
static double* real_data(const mxArray* a) {
#if OFDM_INTERLEAVED
    return mxGetDoubles(a);
#else
    return mxGetPr(a);
#endif
}
/* complex mxArray (n elements, MATLAB order) -> device buffer of the context's type */
static void* to_dev_complex(const mxArray* a, size_t n) {
    size_t i;
    void* h = hostbuf(n * esz());
    for (i = 0; i < n; ++i) {
        double re, im; get_complex(a, i, &re, &im);
        if (g_prec == OFDM_PREC_F64) { ((double*)h)[2 * i] = re; ((double*)h)[2 * i + 1] = im; }
        else { ((float*)h)[2 * i] = (float)re; ((float*)h)[2 * i + 1] = (float)im; }
    }
    void* d = devbuf(n * esz());
    chk(ofdm_h2d(g_ctx, d, h, n * esz()), "h2d");
    return d;
}
static mxArray* from_dev_complex(const void* d, size_t rows, size_t cols) {
    size_t n = rows * cols, i;
    void* h = hostbuf(n * esz());
    mxArray* out;
    chk(ofdm_d2h(g_ctx, h, d, n * esz()), "d2h");
    out = mxCreateDoubleMatrix(rows, cols, mxCOMPLEX);
    for (i = 0; i < n; ++i) {
        if (g_prec == OFDM_PREC_F64) set_complex(out, i, ((double*)h)[2 * i], ((double*)h)[2 * i + 1]);
        else set_complex(out, i, ((float*)h)[2 * i], ((float*)h)[2 * i + 1]);
    }
    return out;
}
/* 0/1 doubles -> packed words on the device */
static uint32_t* to_dev_bits(const mxArray* a, size_t n) {
    size_t i, words = OFDM_BIT_WORDS(n) ? OFDM_BIT_WORDS(n) : 1;
    uint32_t* h = (uint32_t*)hostbuf(words * 4);
    double* p = real_data(a);
    for (i = 0; i < n; ++i) if (p[i] != 0.0) h[i >> 5] |= 1u << (i & 31);
    uint32_t* d = (uint32_t*)devbuf(words * 4);
    chk(ofdm_h2d(g_ctx, d, h, words * 4), "h2d");
    return d;
}
static mxArray* from_dev_bits(const uint32_t* d, size_t n) {   /* 1 x n row of 0/1 doubles */
    size_t i, words = OFDM_BIT_WORDS(n) ? OFDM_BIT_WORDS(n) : 1;
    uint32_t* h = (uint32_t*)hostbuf(words * 4);
    mxArray* out;
    double* p;
    chk(ofdm_d2h(g_ctx, h, d, words * 4), "d2h");
    out = mxCreateDoubleMatrix(1, n, mxREAL);
    p = real_data(out);
    for (i = 0; i < n; ++i) p[i] = (double)((h[i >> 5] >> (i & 31)) & 1u);
    return out;
}
static int32_t* to_i32(const mxArray* a, int* n) {   /* 1-based index vector, kept 1-based for the ABI */
    size_t i, cnt = mxGetNumberOfElements(a);
    int32_t* v = (int32_t*)hostbuf(cnt * 4);
    double* p = real_data(a);
    for (i = 0; i < cnt; ++i) v[i] = (int32_t)llround(p[i]);
    *n = (int)cnt;
    return v;
}
static double* to_cdoubles(const mxArray* a, size_t n) {   /* complex doubles, interleaved, host */
    size_t i;
    double* v = (double*)hostbuf(n * 16);
    for (i = 0; i < n; ++i) get_complex(a, i, &v[2 * i], &v[2 * i + 1]);
    return v;
}
static uint8_t* to_reg(const mxArray* a) {
    size_t i;
    uint8_t* r = (uint8_t*)hostbuf(16);
    if (mxGetNumberOfElements(a) != 15) fail("ofdm:arg:register", "Register must have 15 cells");
    for (i = 0; i < 15; ++i) r[i] = real_data(a)[i] != 0.0;
    return r;
}
static int constellation_id(const mxArray* a) {
    char s[16];
    if (!mxIsChar(a) || mxGetString(a, s, sizeof s)) fail("ofdm:arg:constellation", "constellation must be a char/string name");
    if (!strcmp(s, "BPSK")) return OFDM_BPSK;
    if (!strcmp(s, "QPSK")) return OFDM_QPSK;
    if (!strcmp(s, "8PSK")) return OFDM_8PSK;
    if (!strcmp(s, "16QAM")) return OFDM_16QAM;
    fail("ofdm:arg:constellation", "unknown constellation");
    return 0;
}
static double* dev_doubles(const double* h, size_t n) {
    double* d = (double*)devbuf(n * 8);
    chk(ofdm_h2d(g_ctx, d, h, n * 8), "h2d");
    return d;
}
static mxArray* scalar_from_dev_f64(const double* d) { double v; chk(ofdm_d2h(g_ctx, &v, d, 8), "d2h"); return mxCreateDoubleScalar(v); }
static mxArray* scalar_from_dev_i32(const int32_t* d) { int32_t v; chk(ofdm_d2h(g_ctx, &v, d, 4), "d2h"); return mxCreateDoubleScalar((double)v); }


/* ---- batched / fused ops: the link description travels as ten positional arguments --------------------------------
 *   LINK = Nfft, T_Guard, N_carrier, N_symb, SpF, Constellation, dataCarriers, pilotCarriers, pilotValues, Register
 * (the literals at the top of every reference script, `Task 5/Main_model_Task_5.m:6-46`); matlab/ofdm_link.m packs a
 * struct into this list.  Batches are columns: one serial stream / one stream's bits per column. */
#define N_LINK 10
static void parse_link(const mxArray* const* a, ofdm_link_params* lp) {
    int nd = 0, np = 0;
    memset(lp, 0, sizeof *lp);
    lp->Nfft = (int32_t)mxGetScalar(a[0]); lp->Tg = (int32_t)mxGetScalar(a[1]); lp->N_carrier = (int32_t)mxGetScalar(a[2]);
    lp->S = (int32_t)mxGetScalar(a[3]); lp->SpF = (int32_t)mxGetScalar(a[4]);
    lp->constellation = constellation_id(a[5]);
    lp->data_carriers_host = to_i32(a[6], &nd);
    lp->pilot_carriers_host = to_i32(a[7], &np);
    lp->Nd = nd; lp->Np = np;
    if (lp->S <= 0 || lp->SpF <= 0 || lp->S % lp->SpF) fail("ofdm:arg:link", "N_symb must be a positive multiple of SpF");
    if (mxGetNumberOfElements(a[8]) == (size_t)np * lp->S) lp->pilot_vals_host = to_cdoubles(a[8], (size_t)np * lp->S);
    else if (mxGetNumberOfElements(a[8]) == (size_t)np) {            /* one column: the same pilots in every symbol */
        double* col = to_cdoubles(a[8], (size_t)np);
        double* all = (double*)hostbuf((size_t)np * lp->S * 16);
        int s2;
        for (s2 = 0; s2 < lp->S; ++s2) memcpy(all + (size_t)s2 * np * 2, col, (size_t)np * 16);
        lp->pilot_vals_host = all;
    } else fail("ofdm:arg:pilots", "pilotValues must be Np x N_symb or Np x 1");
    lp->reg0_host = to_reg(a[9]);
    lp->scramble = 1;
}
static int64_t link_stream_bits(const ofdm_link_params* lp) { int bps = 0; ofdm_constellation(lp->constellation, NULL, &bps); return (int64_t)lp->S * lp->Nd * bps; }
/* host matrix of 0/1 doubles, one stream per column (rows = stream_bits, a multiple of 32) -> packed words, host */
static uint32_t* pack_bit_columns(const mxArray* a, size_t bits, size_t B) {
    size_t words = bits / 32, b, i;
    uint32_t* h = (uint32_t*)hostbuf(words * B * 4 + 4);
    const double* p = real_data(a);
    for (b = 0; b < B; ++b)
        for (i = 0; i < bits; ++i) if (p[b * bits + i] != 0.0) h[b * words + (i >> 5)] |= 1u << (i & 31);
    return h;
}

#define NEED(n) do { if (nrhs < (n) + 1) fail("ofdm:arg:count", "too few input arguments"); } while (0)
#define A(i) prhs[(i) + 1]
#define OUT(i, v) do { if ((i) == 0 || nlhs > (i)) plhs[i] = (v); else mxDestroyArray(v); } while (0)

void mexFunction(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    char op[48];
    if (nrhs < 1 || !mxIsChar(prhs[0]) || mxGetString(prhs[0], op, sizeof op)) mexErrMsgIdAndTxt("ofdm:arg:op", "first argument must be the operation name");
    if (!strcmp(op, "precision")) {   /* ofdm_mex('precision','f64'|'f32'): switch the comparison mode */
        char s[8];
        NEED(1);
        if (mxGetString(A(0), s, sizeof s)) mexErrMsgIdAndTxt("ofdm:arg:precision", "expected 'f32' or 'f64'");
        at_exit();
        g_prec = !strcmp(s, "f64") ? OFDM_PREC_F64 : OFDM_PREC_F32;
        return;
    }
    ensure_ctx();

    if (!strcmp(op, "devices")) {   /* ids = ofdm_mex('devices' [, ids]): the 0-based CUDA devices of the six sweep ops */
        if (nrhs > 1) {
            size_t n = mxGetNumberOfElements(A(0)), i;
            int ids[MAX_DEVICES];
            if (!mxIsDouble(A(0)) || mxIsComplex(A(0))) mexErrMsgIdAndTxt("ofdm:devices:type", "device ids must be real doubles");
            if (n == 0) mexErrMsgIdAndTxt("ofdm:devices:empty", "need at least one device id");
            if (n > MAX_DEVICES) mexErrMsgIdAndTxt("ofdm:devices:count", "at most %d device ids", MAX_DEVICES);
            for (i = 0; i < n; ++i) {
                double v = real_data(A(0))[i];
                if (!(v >= 0 && v <= 1e6 && v == floor(v))) mexErrMsgIdAndTxt("ofdm:devices:id", "device ids are 0-based integers >= 0");
                ids[i] = (int)v;
            }
            ofdm_group_destroy(g_group); g_group = NULL;
            memcpy(g_devices, ids, n * sizeof(int));
            g_ndevices = (int)n;
            if (!(g_ndevices == 1 && g_devices[0] == 0) && ofdm_group_create(&g_group, g_devices, g_ndevices, g_prec) != OFDM_OK) {
                g_devices[0] = 0; g_ndevices = 1;                   /* back to the default set */
                mexErrMsgIdAndTxt("ofdm:devices:nodevice", "a device of the set is not an sm_100 GPU of this host; the set is [0] again");
            }
        }
        {
            mxArray* dm = mxCreateDoubleMatrix(1, (size_t)g_ndevices, mxREAL);
            int i;
            for (i = 0; i < g_ndevices; ++i) real_data(dm)[i] = g_devices[i];
            OUT(0, dm);
        }
        return;
    }
    if (!strcmp(op, "Scrambler") || !strcmp(op, "DeScrambler")) {            /* [seq, Register] = f(Register, sequence) */
        NEED(2);
        size_t L = mxGetNumberOfElements(A(1)), i;
        uint8_t* reg = to_reg(A(0));
        uint32_t* in = to_dev_bits(A(1), L);
        uint32_t* out = (uint32_t*)devbuf((OFDM_BIT_WORDS(L) + 1) * 4);
        uint8_t* fr = (uint8_t*)devbuf(16);
        uint8_t frh[15];
        mxArray* r;
        chk((op[0] == 'S' ? ofdm_scramble : ofdm_descramble)(g_ctx, in, out, 1, (int64_t)L, reg, fr), op);
        OUT(0, from_dev_bits(out, L));
        chk(ofdm_d2h(g_ctx, frh, fr, 15), "d2h");
        r = mxCreateDoubleMatrix(1, 15, mxREAL);
        for (i = 0; i < 15; ++i) real_data(r)[i] = frh[i];
        OUT(1, r);
    } else if (!strcmp(op, "constellation_func")) {                          /* [Dictionary, bps] = f(name) */
        NEED(1);
        double tab[32]; int bps = 0, i;
        mxArray* d;
        if (ofdm_constellation(constellation_id(A(0)), tab, &bps)) fail("ofdm:arg:constellation", "unknown constellation");
        d = mxCreateDoubleMatrix(1, (size_t)1 << bps, mxCOMPLEX);
        for (i = 0; i < (1 << bps); ++i) set_complex(d, i, tab[2 * i], tab[2 * i + 1]);
        OUT(0, d);
        OUT(1, mxCreateDoubleScalar(bps));
    } else if (!strcmp(op, "mapping")) {                                     /* [IQ, pad] = f(bits, constellation) */
        NEED(2);
        size_t n = mxGetNumberOfElements(A(0));
        int cid = constellation_id(A(1)), pad = -1, bps = 0;
        ofdm_constellation(cid, NULL, &bps);
        size_t ns = (n + bps - 1) / bps;
        void* iq = devbuf(ns * esz());
        chk(ofdm_map(g_ctx, to_dev_bits(A(0), n), (int64_t)n, cid, iq, &pad), op);
        OUT(0, from_dev_complex(iq, 1, ns));
        OUT(1, mxCreateDoubleScalar(pad));
    } else if (!strcmp(op, "demapping")) {                                   /* bits = f(pad, IQ, Constellation) */
        NEED(3);
        int pad = (int)mxGetScalar(A(0)), cid = constellation_id(A(2)), bps = 0;
        size_t ns = mxGetNumberOfElements(A(1));
        ofdm_constellation(cid, NULL, &bps);
        uint32_t* bits = (uint32_t*)devbuf((OFDM_BIT_WORDS(ns * bps) + 1) * 4);
        chk(ofdm_demap(g_ctx, to_dev_complex(A(1), ns), (int64_t)ns, cid, bits, 0.0, NULL), op);
        OUT(0, from_dev_bits(bits, ns * bps - (pad != -1 ? (size_t)pad : 0)));
    } else if (!strcmp(op, "OFDM_map_carriers")) {   /* grid = f(QAM, N_symb, Nfft, dataCarriers, pilotCarriers, pilotValues) */
        NEED(6);
        int S = (int)mxGetScalar(A(1)), Nfft = (int)mxGetScalar(A(2)), Nd, Np;
        int32_t* dc = to_i32(A(3), &Nd);
        int32_t* pc = to_i32(A(4), &Np);
        size_t npv = mxGetNumberOfElements(A(5));
        int mode = npv == 1 ? 1 : 0;
        if (mode == 0 && npv != (size_t)Np * S) fail("ofdm:arg:pilots", "pilotValues must be Np x N_symb or a scalar");
        void* grid = devbuf((size_t)S * Nfft * esz());
        chk(ofdm_map_carriers(g_ctx, to_dev_complex(A(0), (size_t)Nd * S), 1, S, Nfft, dc, Nd, pc, Np, to_cdoubles(A(5), npv), mode, grid), op);
        OUT(0, from_dev_complex(grid, Nfft, S));
    } else if (!strcmp(op, "OFDM_modulator") || !strcmp(op, "OFDM_demodulator")) {   /* out = f(matrix, T_guard) */
        NEED(2);
        int rows = (int)mxGetM(A(0)), S = (int)mxGetN(A(0)), Tg = (int)mxGetScalar(A(1));
        int mod = op[5] == 'm';
        int Nfft = mod ? rows : rows - Tg, orows = mod ? rows + Tg : Nfft;
        void* out = devbuf((size_t)orows * S * esz());
        void* in = to_dev_complex(A(0), (size_t)rows * S);
        chk(mod ? ofdm_modulate(g_ctx, in, 1, S, Nfft, Tg, out) : ofdm_demodulate(g_ctx, in, 1, S, Nfft, Tg, out), op);
        OUT(0, from_dev_complex(out, orows, S));
    } else if (!strcmp(op, "get_payload")) {                                 /* RX_IQ = f(grid, dataCarriers) */
        NEED(2);
        int Nfft = (int)mxGetM(A(0)), S = (int)mxGetN(A(0)), Nd;
        int32_t* dc = to_i32(A(1), &Nd);
        void* out = devbuf((size_t)Nd * S * esz());
        chk(ofdm_get_payload(g_ctx, to_dev_complex(A(0), (size_t)Nfft * S), 1, S, Nfft, dc, Nd, out), op);
        OUT(0, from_dev_complex(out, Nd, S));
    } else if (!strcmp(op, "add_STO") || !strcmp(op, "add_CFO")) {           /* y = add_STO(y, nSTO) | add_CFO(y, CFO, Nfft) */
        NEED(2);
        size_t L = mxGetNumberOfElements(A(0));
        void* in = to_dev_complex(A(0), L);
        void* out = devbuf(L * esz());
        if (op[4] == 'S') {
            int32_t n = (int32_t)mxGetScalar(A(1));
            int32_t* nd = (int32_t*)devbuf(4);
            chk(ofdm_h2d(g_ctx, nd, &n, 4), "h2d");
            chk(ofdm_add_sto(g_ctx, in, 1, (int64_t)L, nd, out), op);
        } else {
            NEED(3);
            double c = mxGetScalar(A(1));
            chk(ofdm_add_cfo(g_ctx, in, 1, (int64_t)L, dev_doubles(&c, 1), (int)mxGetScalar(A(2)), out), op);
        }
        OUT(0, from_dev_complex(out, L, 1));
    } else if (!strcmp(op, "Noise")) {   /* [IQ_RX, N_var] = Noise(SNR, IQ_TX [, normals (L x 2) | seed]) */
        NEED(2);
        size_t L = mxGetNumberOfElements(A(1)), i;
        double snr = mxGetScalar(A(0));
        void* in = to_dev_complex(A(1), L);
        void* out = devbuf(L * esz());
        double* nv = (double*)devbuf(8);
        void* normals = NULL;
        uint64_t seed = 0;
        if (nrhs >= 4 && mxGetNumberOfElements(A(2)) == 2 * L) {            /* imported realisation: column 1 real, column 2 imaginary */
            double* p = real_data(A(2));
            void* h = hostbuf(2 * L * rsz());
            for (i = 0; i < 2 * L; ++i) { if (g_prec == OFDM_PREC_F64) ((double*)h)[i] = p[i]; else ((float*)h)[i] = (float)p[i]; }
            normals = devbuf(2 * L * rsz());
            chk(ofdm_h2d(g_ctx, normals, h, 2 * L * rsz()), "h2d");
        } else if (nrhs >= 4) seed = (uint64_t)mxGetScalar(A(2));
        chk(ofdm_add_noise(g_ctx, in, 1, (int64_t)L, dev_doubles(&snr, 1), normals, seed, 0, out, nv), op);
        OUT(0, from_dev_complex(out, mxGetM(A(1)), mxGetN(A(1))));
        OUT(1, scalar_from_dev_f64(nv));
    } else if (!strcmp(op, "get_MP_channel_resp")) {                         /* [h, H] = f(channel_taps (K x 2), Nfft) */
        NEED(2);
        int K = (int)mxGetM(A(0)), Nfft = (int)mxGetScalar(A(1)), hl = 0, i;
        double* tp = real_data(A(0));
        double* taps = (double*)hostbuf((size_t)K * 16);
        double* h = (double*)hostbuf(65536 * 8);
        void* H = devbuf((size_t)Nfft * esz());
        mxArray* hm;
        for (i = 0; i < K; ++i) { taps[2 * i] = tp[i]; taps[2 * i + 1] = tp[K + i]; }   /* column-major K x 2 */
        chk(ofdm_mp_channel_resp(g_ctx, taps, K, Nfft, h, 65536, &hl, H), op);
        hm = mxCreateDoubleMatrix(1, hl, mxREAL);
        memcpy(real_data(hm), h, (size_t)hl * 8);
        OUT(0, hm);
        OUT(1, from_dev_complex(H, 1, Nfft));
    } else if (!strcmp(op, "apply_channel")) {                               /* y = conv(x, h.', 'full')(1:numel(x)) */
        NEED(2);
        size_t L = mxGetNumberOfElements(A(0)), D = mxGetNumberOfElements(A(1));
        void* out = devbuf(L * esz());
        chk(ofdm_apply_fir(g_ctx, to_dev_complex(A(0), L), 1, (int64_t)L, to_dev_complex(A(1), D), (int)D, 0, out), op);
        OUT(0, from_dev_complex(out, L, 1));
    } else if (!strcmp(op, "AutoCorrFunction")) {                            /* [AutoCorr, TgPosition, FreqOffset] = f(Rx, W, Nfft) */
        NEED(3);
        size_t L = mxGetNumberOfElements(A(0));
        int W = (int)mxGetScalar(A(1)), Nfft = (int)mxGetScalar(A(2));
        size_t no = L - W - Nfft;
        void* ac = devbuf(no * esz());
        int32_t* tg = (int32_t*)devbuf(4);
        double* fo = (double*)devbuf(8);
        chk(ofdm_cp_autocorr(g_ctx, to_dev_complex(A(0), L), 1, (int64_t)L, W, Nfft, ac, tg, fo, NULL), op);
        OUT(0, from_dev_complex(ac, 1, no));
        OUT(1, scalar_from_dev_i32(tg));
        OUT(2, scalar_from_dev_f64(fo));
    } else if (!strcmp(op, "remove_IFO")) {                                  /* [fixed, IFO] = f(rx, Nfft) */
        NEED(2);
        size_t L = mxGetNumberOfElements(A(0));
        void* out = devbuf(L * esz());
        int32_t* ifo = (int32_t*)devbuf(4);
        int32_t k;
        chk(ofdm_remove_ifo(g_ctx, to_dev_complex(A(0), L), 1, (int64_t)L, (int)mxGetScalar(A(1)), out, ifo), op);
        chk(ofdm_d2h(g_ctx, &k, ifo, 4), "d2h");
        if (k < 0) fail("ofdm:remove_IFO:empty", "no spectrum bin above 0.77 (inds(1) on an empty find)");
        OUT(0, from_dev_complex(out, L, 1));
        OUT(1, mxCreateDoubleScalar(k));
    } else if (!strcmp(op, "fine_sync")) {               /* out = f(rx, pilotCarriers, pilotValues, time_desync, freq_desync) */
        NEED(5);
        int Nfft = (int)mxGetM(A(0)), S = (int)mxGetN(A(0)), Np;
        int32_t* pc = to_i32(A(1), &Np);
        void* out = devbuf((size_t)Nfft * S * esz());
        chk(ofdm_fine_sync(g_ctx, to_dev_complex(A(0), (size_t)Nfft * S), 1, S, Nfft, pc, Np, to_cdoubles(A(2), (size_t)Np * S),
                           mxGetScalar(A(3)) != 0, mxGetScalar(A(4)) != 0, out, NULL, NULL), op);
        OUT(0, from_dev_complex(out, Nfft, S));
    } else if (!strcmp(op, "estimate_channel")) {        /* [H_est, Hp] = f(rx, allCarriers, pilotCarriers, pilotValues) */
        NEED(4);
        int Nfft = (int)mxGetM(A(0)), S = (int)mxGetN(A(0)), Nq, Np;
        int32_t* ac = to_i32(A(1), &Nq);
        int32_t* pc = to_i32(A(2), &Np);
        void* H = devbuf((size_t)Nq * esz());
        void* Hp = devbuf((size_t)Np * esz());
        chk(ofdm_estimate_channel(g_ctx, to_dev_complex(A(0), (size_t)Nfft * S), 1, S, Nfft, ac, Nq, pc, Np, to_cdoubles(A(3), (size_t)Np * S), H, Hp), op);
        OUT(0, from_dev_complex(H, 1, Nq));
        OUT(1, from_dev_complex(Hp, Np, 1));
    } else if (!strcmp(op, "LS_CE")) {                                       /* H_LS = f(Y, Xp, pilot_loc, N_carrier) */
        NEED(4);
        int Nfft = (int)mxGetM(A(0)), S = (int)mxGetN(A(0)), Np, Nc = (int)mxGetScalar(A(3));
        int32_t* pc = to_i32(A(2), &Np);
        void* H = devbuf((size_t)Nc * esz());
        chk(ofdm_ls_ce(g_ctx, to_dev_complex(A(0), (size_t)Nfft * S), 1, S, Nfft, pc, Np, to_cdoubles(A(1), Np), Nc, H), op);
        OUT(0, from_dev_complex(H, 1, Nc));
    } else if (!strcmp(op, "MMSE_CE")) {                 /* H = f(Y, Xp, pilot_loc, Nfft, N_carrier, h, SNR) */
        NEED(7);
        int Nfft = (int)mxGetM(A(0)), S = (int)mxGetN(A(0)), Np, Nc = (int)mxGetScalar(A(4));
        int32_t* pc = to_i32(A(2), &Np);
        size_t hl = mxGetNumberOfElements(A(5));
        double snr = mxGetScalar(A(6));
        void* H = devbuf((size_t)Nc * esz());
        chk(ofdm_mmse_ce(g_ctx, to_dev_complex(A(0), (size_t)Nfft * S), 1, S, Nfft, pc, Np, to_cdoubles(A(1), Np), Nc, to_dev_complex(A(5), hl), (int)hl,
                         dev_doubles(&snr, 1), H), op);
        OUT(0, from_dev_complex(H, 1, Nc));
    } else if (!strcmp(op, "interpolate")) {                                 /* H = f(H, pilot_loc, Nfft, method) */
        NEED(4);
        int Np, N = (int)mxGetScalar(A(2));
        int32_t* pc = to_i32(A(1), &Np);
        char m[16];
        void* H = devbuf((size_t)N * esz());
        if (mxGetString(A(3), m, sizeof m)) fail("ofdm:arg:method", "method must be a string");
        chk(ofdm_interpolate(g_ctx, to_dev_complex(A(0), Np), 1, pc, Np, N, (m[0] == 'l' || m[0] == 'L') ? OFDM_INTERP_LINEAR : OFDM_INTERP_SPLINE, H), op);
        OUT(0, from_dev_complex(H, 1, N));
    } else if (!strcmp(op, "equalize_signal")) {                             /* out = f(OFDM_demod, Hest, N_carrier) */
        NEED(3);
        int Nfft = (int)mxGetM(A(0)), S = (int)mxGetN(A(0)), Nc = (int)mxGetScalar(A(2));
        size_t hn = mxGetNumberOfElements(A(1));
        void* out = devbuf((size_t)Nfft * S * esz());
        chk(ofdm_equalize(g_ctx, to_dev_complex(A(0), (size_t)Nfft * S), 1, S, Nfft, to_dev_complex(A(1), hn), (int)hn, Nc, out), op);
        OUT(0, from_dev_complex(out, Nfft, S));
    } else if (!strcmp(op, "OMP_estimate") || !strcmp(op, "MP_estimate")) {  /* [H, h, index] = f(Y, sensing_matrix, Nfft, taps [, SNR]) */
        NEED(4);
        int Np = (int)mxGetM(A(1)), Ld = (int)mxGetN(A(1)), Nfft = (int)mxGetScalar(A(2)), K = (int)mxGetScalar(A(3));
        int omp = op[0] == 'O';
        void* H = devbuf((size_t)Nfft * esz());
        void* h = devbuf((size_t)Nfft * esz());
        int32_t* idx = (int32_t*)devbuf((size_t)K * 4 + 4);
        int32_t* it = (int32_t*)devbuf(4);
        void* y = to_dev_complex(A(0), Np);
        void* Ad = to_dev_complex(A(1), (size_t)Np * Ld);
        if (omp) chk(ofdm_omp(g_ctx, y, 1, Np, Ad, Ld, NULL, Nfft, K, H, h, idx, it), op);
        else chk(ofdm_mp(g_ctx, y, 1, Np, Ad, Ld, NULL, Nfft, K, H, h, idx), op);
        OUT(0, from_dev_complex(H, 1, Nfft));
        OUT(1, omp ? from_dev_complex(h, 1, Nfft) : from_dev_complex(h, Nfft, 1));   /* row for OMP, column for MP, as the reference */
        if (omp) {
            int32_t n, ih[32], i;
            mxArray* ix;
            chk(ofdm_d2h(g_ctx, &n, it, 4), "d2h");
            chk(ofdm_d2h(g_ctx, ih, idx, (size_t)K * 4), "d2h");
            ix = mxCreateDoubleMatrix(1, n, mxREAL);
            for (i = 0; i < n; ++i) real_data(ix)[i] = ih[i];
            OUT(2, ix);
        }
    } else if (!strcmp(op, "BER_func")) {                                    /* BER = f(Bit_Tx, Bit_Rx) */
        NEED(2);
        size_t n = mxGetNumberOfElements(A(0));
        int64_t* c = (int64_t*)devbuf(16);
        int64_t ch[2];
        chk(ofdm_memset(g_ctx, c, 0, 16), "memset");
        chk(ofdm_ber_count(g_ctx, to_dev_bits(A(0), n), to_dev_bits(A(1), n), (int64_t)n, c), op);
        chk(ofdm_d2h(g_ctx, ch, c, 16), "d2h");
        OUT(0, mxCreateDoubleScalar((double)ch[0] / (double)ch[1]));
    } else if (!strcmp(op, "MER_func")) {                                    /* MER = f(IQ_RX, Constellation) */
        NEED(2);
        size_t n = mxGetNumberOfElements(A(0));
        double* s = (double*)devbuf(16);
        double sh[2];
        chk(ofdm_memset(g_ctx, s, 0, 16), "memset");
        chk(ofdm_mer(g_ctx, to_dev_complex(A(0), n), (int64_t)n, constellation_id(A(1)), s), op);
        chk(ofdm_d2h(g_ctx, sh, s, 16), "d2h");
        OUT(0, mxCreateDoubleScalar(10.0 * log10(sh[0] / sh[1])));
    } else if (!strcmp(op, "calculatePAPR")) {                               /* PAPR = f(OFDM_signal) */
        NEED(1);
        size_t n = mxGetNumberOfElements(A(0));
        double* d = (double*)devbuf(8);
        chk(ofdm_papr(g_ctx, to_dev_complex(A(0), n), 1, (int64_t)n, d), op);
        OUT(0, scalar_from_dev_f64(d));
    } else if (!strcmp(op, "calculate_window_PAPR")) {                       /* PAPRs (1 x L-Nfft+1) = f(Tx_OFDM_Signal, Nfft) */
        NEED(2);
        size_t n = mxGetNumberOfElements(A(0)), i;
        int W = (int)mxGetScalar(A(1));
        if (W < 1 || (size_t)W > n) fail("ofdm:calculate_window_PAPR:size", "Nfft must be in 1..length(signal)");
        size_t no = n - (size_t)W + 1;
        void* d = devbuf(rsz() * no);
        void* h = hostbuf(rsz() * no);
        chk(ofdm_window_papr(g_ctx, to_dev_complex(A(0), n), 1, (int64_t)n, W, d), op);
        chk(ofdm_d2h(g_ctx, h, d, rsz() * no), "d2h");
        mxArray* o = mxCreateDoubleMatrix(1, no, mxREAL);
        for (i = 0; i < no; ++i) real_data(o)[i] = g_prec == OFDM_PREC_F64 ? ((double*)h)[i] : (double)((float*)h)[i];
        OUT(0, o);
    } else if (!strcmp(op, "calculateCCDF")) {                               /* [PAPR_ccdf, CCDF] = f(PAPR_values): column vectors as ecdf */
        NEED(1);
        size_t n = mxGetNumberOfElements(A(0)), i;
        if (n < 1) fail("ofdm:calculateCCDF:size", "empty input");
        void* hv = hostbuf(rsz() * n);
        for (i = 0; i < n; ++i) { double v = real_data(A(0))[i]; if (g_prec == OFDM_PREC_F64) ((double*)hv)[i] = v; else ((float*)hv)[i] = (float)v; }
        void* dv = devbuf(rsz() * n);
        void* dx = devbuf(rsz() * (n + 1));
        void* dc = devbuf(rsz() * (n + 1));
        int64_t* dn = (int64_t*)devbuf(8);
        int64_t k = 0;
        chk(ofdm_h2d(g_ctx, dv, hv, rsz() * n), "h2d");
        chk(ofdm_ccdf(g_ctx, dv, (int64_t)n, dx, dc, dn), op);
        chk(ofdm_d2h(g_ctx, &k, dn, 8), "d2h");
        void* hx = hostbuf(rsz() * (size_t)k);
        void* hc = hostbuf(rsz() * (size_t)k);
        chk(ofdm_d2h(g_ctx, hx, dx, rsz() * (size_t)k), "d2h");
        chk(ofdm_d2h(g_ctx, hc, dc, rsz() * (size_t)k), "d2h");
        mxArray* ox = mxCreateDoubleMatrix((size_t)k, 1, mxREAL);
        mxArray* oc = mxCreateDoubleMatrix((size_t)k, 1, mxREAL);
        for (i = 0; i < (size_t)k; ++i) {
            real_data(ox)[i] = g_prec == OFDM_PREC_F64 ? ((double*)hx)[i] : (double)((float*)hx)[i];
            real_data(oc)[i] = g_prec == OFDM_PREC_F64 ? ((double*)hc)[i] : (double)((float*)hc)[i];
        }
        OUT(0, ox);
        OUT(1, oc);
    } else if (!strcmp(op, "tx_chain")) {                 /* Tx (L x B) = tx_chain(LINK..., bits (stream_bits x B)) */
        NEED(N_LINK + 1);
        ofdm_link_params lp;
        parse_link(&A(0), &lp);
        int64_t sb = link_stream_bits(&lp);
        size_t B, L = (size_t)lp.S * (lp.Nfft + lp.Tg);
        if (sb % 32 || mxGetM(A(N_LINK)) != (size_t)sb) fail("ofdm:tx_chain:bits", "bits must be stream_bits x B with stream_bits = N_symb*Nd*bps divisible by 32");
        B = mxGetN(A(N_LINK));
        uint32_t* hb = pack_bit_columns(A(N_LINK), (size_t)sb, B);
        uint32_t* db = (uint32_t*)devbuf((size_t)sb / 8 * B + 4);
        void* tx = devbuf(L * B * esz());
        chk(ofdm_h2d(g_ctx, db, hb, (size_t)sb / 8 * B), "h2d");
        chk(ofdm_tx_chain(g_ctx, &lp, db, (int64_t)B, tx), op);
        OUT(0, from_dev_complex(tx, L, B));
    } else if (!strcmp(op, "channel_t5")) {               /* Rx = channel_t5(Tx (L x B), SNR_dB (scalar | 1 x B | []), h (FIR | []), seed) */
        NEED(4);
        size_t L = mxGetM(A(0)), B = mxGetN(A(0)), ns = mxGetNumberOfElements(A(1)), D = mxGetNumberOfElements(A(2)), b;
        double* snr = NULL;
        if (ns) {
            double* sh = (double*)hostbuf(B * 8);
            if (ns != 1 && ns != B) fail("ofdm:channel_t5:snr", "SNR_dB must be a scalar, 1 x B or empty");
            for (b = 0; b < B; ++b) sh[b] = real_data(A(1))[ns == 1 ? 0 : b];
            snr = dev_doubles(sh, B);
        }
        void* rx = devbuf(L * B * esz());
        chk(ofdm_channel_t5(g_ctx, to_dev_complex(A(0), L * B), (int64_t)B, (int64_t)L, snr, NULL, (uint64_t)mxGetScalar(A(3)), 0,
                            D ? to_dev_complex(A(2), D) : NULL, (int)D, rx), op);
        OUT(0, from_dev_complex(rx, L, B));
    } else if (!strcmp(op, "channel_t4")) {               /* Rx = channel_t4(Tx (L x B), SNR_dB (scalar | 1 x B), STO (scalar | 1 x B), CFO (scalar | 1 x B), Nfft, h (FIR), seed) */
        NEED(7);                                          /* Noise -> add_STO -> add_CFO -> conv(h), `Task 4/Main_model_Task_4.m:95,103,110,263-264`, in one pass */
        size_t L = mxGetM(A(0)), B = mxGetN(A(0)), D = mxGetNumberOfElements(A(5)), b, k;
        double* hd = (double*)hostbuf(B * 8 * 2);
        int32_t* hs = (int32_t*)hostbuf(B * 4);
        double* dv[2];
        int32_t* sto_d;
        for (k = 1; k <= 3; ++k) {
            size_t ne = mxGetNumberOfElements(A(k));
            if (ne != 1 && ne != B) fail("ofdm:channel_t4:arg", "SNR_dB, STO and CFO must be scalars or 1 x B");
        }
        if (!D) fail("ofdm:channel_t4:h", "h must hold at least one tap (1 for no multipath)");
        for (b = 0; b < B; ++b) hd[b] = real_data(A(1))[mxGetNumberOfElements(A(1)) == 1 ? 0 : b];
        dv[0] = dev_doubles(hd, B);
        for (b = 0; b < B; ++b) hd[b] = real_data(A(3))[mxGetNumberOfElements(A(3)) == 1 ? 0 : b];
        dv[1] = dev_doubles(hd, B);
        for (b = 0; b < B; ++b) hs[b] = (int32_t)real_data(A(2))[mxGetNumberOfElements(A(2)) == 1 ? 0 : b];
        sto_d = (int32_t*)devbuf(B * 4);
        chk(ofdm_h2d(g_ctx, sto_d, hs, B * 4), "h2d");
        void* rx = devbuf(L * B * esz());
        chk(ofdm_channel_t4_p(g_ctx, to_dev_complex(A(0), L * B), (int64_t)B, (int64_t)L, dv[0], NULL, NULL, (uint64_t)mxGetScalar(A(6)), 0, sto_d, dv[1],
                              (int)mxGetScalar(A(4)), to_dev_complex(A(5), D), (int)D, rx), op);
        OUT(0, from_dev_complex(rx, L, B));
    } else if (!strcmp(op, "rx_chain_t5")) {   /* [bits (stream_bits x B), H (N_carrier x B), counts (1 x 3)] = rx_chain_t5(LINK..., Rx (L x B), tx_bits | [], near_eps) */
        NEED(N_LINK + 3);
        ofdm_link_params lp;
        parse_link(&A(0), &lp);
        int64_t sb = link_stream_bits(&lp);
        size_t L = (size_t)lp.S * (lp.Nfft + lp.Tg), B = mxGetN(A(N_LINK)), i, b, words = (size_t)sb / 32;
        int has_tx = mxGetNumberOfElements(A(N_LINK + 1)) != 0;
        if (sb % 32) fail("ofdm:rx_chain_t5:bits", "stream_bits must be divisible by 32");
        if (mxGetM(A(N_LINK)) != L) fail("ofdm:rx_chain_t5:size", "Rx must be (N_symb*(Nfft+T_Guard)) x B");
        if (has_tx && (mxGetM(A(N_LINK + 1)) != (size_t)sb || mxGetN(A(N_LINK + 1)) != B)) fail("ofdm:rx_chain_t5:bits", "tx_bits must be stream_bits x B");
        /* host buffers in the context's type; the library chunks and overlaps H2D / kernel / D2H itself */
        void* rxh = hostbuf(L * B * esz());
        for (i = 0; i < L * B; ++i) {
            double re, im; get_complex(A(N_LINK), i, &re, &im);
            if (g_prec == OFDM_PREC_F64) { ((double*)rxh)[2 * i] = re; ((double*)rxh)[2 * i + 1] = im; }
            else { ((float*)rxh)[2 * i] = (float)re; ((float*)rxh)[2 * i + 1] = (float)im; }
        }
        uint32_t* txh = has_tx ? pack_bit_columns(A(N_LINK + 1), (size_t)sb, B) : NULL;
        uint32_t* obh = (uint32_t*)hostbuf(words * B * 4 + 4);
        void* Hh = hostbuf((size_t)lp.N_carrier * B * esz());
        int64_t cnt[3] = {0, 0, 0};
        chk(ofdm_rx_chain_t5_host_eps(g_ctx, &lp, rxh, (int64_t)B, txh, obh, Hh, cnt, 0, mxGetScalar(A(N_LINK + 2))), op);
        mxArray* ob = mxCreateDoubleMatrix((size_t)sb, B, mxREAL);
        for (b = 0; b < B; ++b)
            for (i = 0; i < (size_t)sb; ++i) real_data(ob)[b * (size_t)sb + i] = (double)((obh[b * words + (i >> 5)] >> (i & 31)) & 1u);
        OUT(0, ob);
        mxArray* Hm = mxCreateDoubleMatrix((size_t)lp.N_carrier, B, mxCOMPLEX);
        for (i = 0; i < (size_t)lp.N_carrier * B; ++i) {
            if (g_prec == OFDM_PREC_F64) set_complex(Hm, i, ((double*)Hh)[2 * i], ((double*)Hh)[2 * i + 1]);
            else set_complex(Hm, i, ((float*)Hh)[2 * i], ((float*)Hh)[2 * i + 1]);
        }
        OUT(1, Hm);
        mxArray* cm = mxCreateDoubleMatrix(1, 3, mxREAL);
        for (i = 0; i < 3; ++i) real_data(cm)[i] = (double)cnt[i];
        OUT(2, cm);
    } else if (!strcmp(op, "sweep_ber")) {   /* counts (n_snr x 4) = sweep_ber(LINK..., snrs, streams_per_point, taps (K x 2 | []), chain, seed, near_eps) */
        NEED(N_LINK + 6);
        ofdm_link_params lp;
        ofdm_sweep_params sp;
        char chain[16];
        parse_link(&A(0), &lp);
        memset(&sp, 0, sizeof sp);
        size_t n = mxGetNumberOfElements(A(N_LINK)), i;
        int K = (int)mxGetM(A(N_LINK + 2));
        if (!n) fail("ofdm:sweep_ber:snr", "need at least one SNR point");
        if (mxGetString(A(N_LINK + 3), chain, sizeof chain)) fail("ofdm:sweep_ber:chain", "chain must be 'task5' or 'task4'");
        sp.chain = !strcmp(chain, "task4") ? OFDM_SWEEP_TASK4 : OFDM_SWEEP_TASK5;
        sp.n_snr = (int32_t)n;
        sp.snr_db_host = real_data(A(N_LINK));
        sp.streams_per_point = (int64_t)mxGetScalar(A(N_LINK + 1));
        sp.rank = 0; sp.world = 1;
        sp.seed = (uint64_t)mxGetScalar(A(N_LINK + 4));
        sp.near_eps = mxGetScalar(A(N_LINK + 5));
        sp.sto_max = lp.Nfft + lp.Tg; sp.cfo_int_max = 30;            /* `Main_model_Task_4.m:101,108` */
        if (mxGetNumberOfElements(A(N_LINK + 2))) {
            double* tp = real_data(A(N_LINK + 2));
            double* taps = (double*)hostbuf((size_t)K * 16);
            int k2;
            if (mxGetN(A(N_LINK + 2)) != 2) fail("ofdm:sweep_ber:taps", "channel_taps must be K x 2 (delay, amplitude)");
            for (k2 = 0; k2 < K; ++k2) { taps[2 * k2] = tp[k2]; taps[2 * k2 + 1] = tp[K + k2]; }
            sp.taps_host = taps; sp.n_taps = K;
        }
        int64_t* ch = (int64_t*)hostbuf(n * 32);
        if (sweep_group()) chk_group(ofdm_group_sweep_ber(g_group, &lp, &sp, ch), op);
        else {
            int64_t* cd = (int64_t*)devbuf(n * 32);
            chk(ofdm_memset(g_ctx, cd, 0, n * 32), "memset");
            chk(ofdm_sweep_ber(g_ctx, &lp, &sp, cd), op);
            chk(ofdm_d2h(g_ctx, ch, cd, n * 32), "d2h");
        }
        mxArray* cm = mxCreateDoubleMatrix(n, 4, mxREAL);
        for (i = 0; i < n; ++i) { int j; for (j = 0; j < 4; ++j) real_data(cm)[(size_t)j * n + i] = (double)ch[4 * i + j]; }
        OUT(0, cm);
    } else if (!strcmp(op, "sweep_mse")) {   /* [MSE (n_snr x 4), per_stream (spp x 4*n_snr), counts (n_snr x 2)] =
                                                 sweep_mse(LINK..., snrs, streams_per_point, taps (K x 2), seed, tie_eps [, Ldict]);
                                                 dataCarriers may be [] (the pilot-only comb-1 layout) */
        NEED(N_LINK + 5);
        ofdm_link_params lp;
        ofdm_sweep_params sp;
        parse_link(&A(0), &lp);
        memset(&sp, 0, sizeof sp);
        size_t n = mxGetNumberOfElements(A(N_LINK)), i;
        int K = (int)mxGetM(A(N_LINK + 2)), k2, e;
        if (!n) fail("ofdm:sweep_mse:snr", "need at least one SNR point");
        if (!K || mxGetN(A(N_LINK + 2)) != 2) fail("ofdm:sweep_mse:taps", "channel_taps must be K x 2 (delay, amplitude)");
        if (lp.Np < 2) fail("ofdm:sweep_mse:pilots", "need at least two pilots");
        sp.chain = OFDM_SWEEP_TASK5;
        sp.n_snr = (int32_t)n;
        sp.snr_db_host = real_data(A(N_LINK));
        sp.streams_per_point = (int64_t)mxGetScalar(A(N_LINK + 1));
        sp.rank = 0; sp.world = 1;
        sp.seed = (uint64_t)mxGetScalar(A(N_LINK + 3));
        sp.near_eps = mxGetScalar(A(N_LINK + 4));
        double* tp = real_data(A(N_LINK + 2));
        double* taps = (double*)hostbuf((size_t)K * 16);
        for (k2 = 0; k2 < K; ++k2) { taps[2 * k2] = tp[k2]; taps[2 * k2 + 1] = tp[K + k2]; }
        sp.taps_host = taps; sp.n_taps = K;
        /* Ldict: the script's ceil(N_carrier / comb) (`Main_model_Task_5.m:182-190`) unless given */
        int comb = lp.pilot_carriers_host[1] - lp.pilot_carriers_host[0];
        int Ldict = nrhs > N_LINK + 6 ? (int)mxGetScalar(A(N_LINK + 5)) : (comb > 0 ? (lp.N_carrier + comb - 1) / comb : 0);
        size_t spp = (size_t)(sp.streams_per_point > 0 ? sp.streams_per_point : 0), cells = n * 4 * spp;
        double* mh = (double*)hostbuf(cells * 8 + 8);
        int64_t* ch = (int64_t*)hostbuf(n * 16);
        if (sweep_group()) chk_group(ofdm_group_sweep_mse(g_group, &lp, &sp, Ldict, mh, ch), op);
        else {
            double* md = (double*)devbuf(cells * 8 + 8);
            int64_t* cd = (int64_t*)devbuf(n * 16);
            chk(ofdm_memset(g_ctx, md, 0, cells * 8), "memset");
            chk(ofdm_memset(g_ctx, cd, 0, n * 16), "memset");
            chk(ofdm_sweep_mse(g_ctx, &lp, &sp, Ldict, md, cd), op);
            chk(ofdm_d2h(g_ctx, mh, md, cells * 8), "d2h");
            chk(ofdm_d2h(g_ctx, ch, cd, n * 16), "d2h");
        }
        mxArray* mm = mxCreateDoubleMatrix(n, 4, mxREAL);           /* mean over the streams of each point */
        for (i = 0; i < n; ++i)
            for (e = 0; e < 4; ++e) {
                double s = 0; size_t j;
                for (j = 0; j < spp; ++j) s += mh[(i * 4 + e) * spp + j];
                real_data(mm)[(size_t)e * n + i] = s / (double)spp;
            }
        OUT(0, mm);
        mxArray* pm = mxCreateDoubleMatrix(spp, 4 * n, mxREAL);     /* reshape(per_stream, spp, 4, n_snr) in MATLAB */
        memcpy(real_data(pm), mh, cells * 8);
        OUT(1, pm);
        mxArray* cm = mxCreateDoubleMatrix(n, 2, mxREAL);
        for (i = 0; i < n; ++i) { real_data(cm)[i] = (double)ch[2 * i]; real_data(cm)[n + i] = (double)ch[2 * i + 1]; }
        OUT(2, cm);
    } else if (!strcmp(op, "sweep_sync")) {   /* [rec (spp x 9*n_snr), counts (n_snr x 4)] =
                                                 sweep_sync(LINK..., snrs, streams_per_point, taps (K x 2, [] = none), seed, sto, cfo,
                                                 [time_desync freq_desync mp_desync] [, sto_max, cfo_int_max]);
                                                 sto < 0: STO / CFO drawn as sweep_ber (sto_max defaults to Nfft + T_Guard, cfo_int_max
                                                 to 30); else every stream gets sto and cfo */
        NEED(N_LINK + 7);
        ofdm_link_params lp;
        ofdm_sync_params sp;
        parse_link(&A(0), &lp);
        memset(&sp, 0, sizeof sp);
        size_t n = mxGetNumberOfElements(A(N_LINK)), i;
        int K = (int)mxGetM(A(N_LINK + 2)), k2;
        if (!n) fail("ofdm:sweep_sync:snr", "need at least one SNR point");
        if (K && mxGetN(A(N_LINK + 2)) != 2) fail("ofdm:sweep_sync:taps", "channel_taps must be K x 2 (delay, amplitude) or []");
        if (mxGetNumberOfElements(A(N_LINK + 6)) != 3) fail("ofdm:sweep_sync:flags", "flags must be [time_desync freq_desync mp_desync]");
        sp.n_snr = (int32_t)n;
        sp.snr_db_host = real_data(A(N_LINK));
        sp.streams_per_point = (int64_t)mxGetScalar(A(N_LINK + 1));
        sp.rank = 0; sp.world = 1;
        sp.seed = (uint64_t)mxGetScalar(A(N_LINK + 3));
        if (K) {
            double* tp = real_data(A(N_LINK + 2));
            double* taps = (double*)hostbuf((size_t)K * 16);
            for (k2 = 0; k2 < K; ++k2) { taps[2 * k2] = tp[k2]; taps[2 * k2 + 1] = tp[K + k2]; }
            sp.taps_host = taps; sp.n_taps = K;
        }
        const double sto = mxGetScalar(A(N_LINK + 4));
        sp.sto_mode = sto < 0 ? 0 : 1;
        sp.sto_fixed = sto < 0 ? 0 : (int32_t)sto;
        sp.cfo_fixed = mxGetScalar(A(N_LINK + 5));
        sp.sto_max = nrhs > N_LINK + 8 ? (int32_t)mxGetScalar(A(N_LINK + 7)) : lp.Nfft + lp.Tg;
        sp.cfo_int_max = nrhs > N_LINK + 9 ? (int32_t)mxGetScalar(A(N_LINK + 8)) : 30;
        const double* fl = real_data(A(N_LINK + 6));
        sp.time_desync = fl[0] != 0; sp.freq_desync = fl[1] != 0; sp.mp_desync = fl[2] != 0;
        size_t spp = (size_t)(sp.streams_per_point > 0 ? sp.streams_per_point : 0), cells = n * 9 * spp;
        int64_t* ch = (int64_t*)hostbuf(n * 32);
        mxArray* rm = mxCreateDoubleMatrix(spp, 9 * n, mxREAL);     /* reshape(rec, spp, 9, n_snr) in MATLAB */
        if (sweep_group()) chk_group(ofdm_group_sweep_sync(g_group, &lp, &sp, cells ? real_data(rm) : (double*)hostbuf(8), ch), op);
        else {
            double* rd = (double*)devbuf(cells * 8 + 8);
            int64_t* cd = (int64_t*)devbuf(n * 32);
            chk(ofdm_memset(g_ctx, rd, 0, cells * 8), "memset");
            chk(ofdm_memset(g_ctx, cd, 0, n * 32), "memset");
            chk(ofdm_sweep_sync(g_ctx, &lp, &sp, rd, cd), op);
            chk(ofdm_d2h(g_ctx, real_data(rm), rd, cells * 8), "d2h");
            chk(ofdm_d2h(g_ctx, ch, cd, n * 32), "d2h");
        }
        OUT(0, rm);
        mxArray* cm = mxCreateDoubleMatrix(n, 4, mxREAL);
        for (i = 0; i < n; ++i) { int j; for (j = 0; j < 4; ++j) real_data(cm)[(size_t)j * n + i] = (double)ch[4 * i + j]; }
        OUT(1, cm);
    } else if (!strcmp(op, "sweep_mer")) {    /* [mer (spp x 2*n_points), counts (n_points x 3)] =
                                                 sweep_mer(LINK..., constellations (ids 1..4, one per point), snrs (one per point),
                                                 streams_per_point, taps (K x 2, [] = none), seed, sto, cfo, pilot_scale, near_eps);
                                                 sto / cfo: one value for every point or one per point */
        NEED(N_LINK + 9);
        ofdm_link_params lp;
        ofdm_mer_params mp;
        parse_link(&A(0), &lp);
        memset(&mp, 0, sizeof mp);
        size_t n = mxGetNumberOfElements(A(N_LINK + 1)), i;
        int K = (int)mxGetM(A(N_LINK + 3)), k2;
        if (!n) fail("ofdm:sweep_mer:snr", "need at least one point");
        if (mxGetNumberOfElements(A(N_LINK)) != n) fail("ofdm:sweep_mer:points", "need one constellation per SNR point");
        if (K && mxGetN(A(N_LINK + 3)) != 2) fail("ofdm:sweep_mer:taps", "channel_taps must be K x 2 (delay, amplitude) or []");
        size_t ns = mxGetNumberOfElements(A(N_LINK + 5)), nc = mxGetNumberOfElements(A(N_LINK + 6));
        if ((ns != 1 && ns != n) || (nc != 1 && nc != n)) fail("ofdm:sweep_mer:impairments", "sto and cfo take one value or one per point");
        int32_t* cons = (int32_t*)hostbuf(n * 8);
        int32_t* nsto = cons + n;
        double* cfo = (double*)hostbuf(n * 8);
        for (i = 0; i < n; ++i) {
            cons[i] = (int32_t)real_data(A(N_LINK))[i];
            nsto[i] = (int32_t)real_data(A(N_LINK + 5))[ns == 1 ? 0 : i];
            cfo[i] = real_data(A(N_LINK + 6))[nc == 1 ? 0 : i];
        }
        mp.n_points = (int32_t)n;
        mp.constellation_host = cons;
        mp.snr_db_host = real_data(A(N_LINK + 1));
        mp.streams_per_point = (int64_t)mxGetScalar(A(N_LINK + 2));
        mp.rank = 0; mp.world = 1;
        mp.seed = (uint64_t)mxGetScalar(A(N_LINK + 4));
        if (K) {
            double* tp = real_data(A(N_LINK + 3));
            double* taps = (double*)hostbuf((size_t)K * 16);
            for (k2 = 0; k2 < K; ++k2) { taps[2 * k2] = tp[k2]; taps[2 * k2 + 1] = tp[K + k2]; }
            mp.taps_host = taps; mp.n_taps = K;
        }
        mp.nsto_host = nsto;
        mp.cfo_host = cfo;
        mp.pilot_scale = mxGetScalar(A(N_LINK + 7));
        mp.near_eps = mxGetScalar(A(N_LINK + 8));
        size_t spp = (size_t)(mp.streams_per_point > 0 ? mp.streams_per_point : 0), cells = n * 2 * spp;
        int64_t* ch = (int64_t*)hostbuf(n * 24);
        mxArray* mm = mxCreateDoubleMatrix(spp, 2 * n, mxREAL);     /* reshape(mer, spp, 2, n_points) in MATLAB */
        if (sweep_group()) chk_group(ofdm_group_sweep_mer(g_group, &lp, &mp, cells ? real_data(mm) : (double*)hostbuf(8), ch), op);
        else {
            double* md = (double*)devbuf(cells * 8 + 8);
            int64_t* cd = (int64_t*)devbuf(n * 24);
            chk(ofdm_memset(g_ctx, md, 0, cells * 8), "memset");
            chk(ofdm_memset(g_ctx, cd, 0, n * 24), "memset");
            chk(ofdm_sweep_mer(g_ctx, &lp, &mp, md, cd), op);
            chk(ofdm_d2h(g_ctx, real_data(mm), md, cells * 8), "d2h");
            chk(ofdm_d2h(g_ctx, ch, cd, n * 24), "d2h");
        }
        OUT(0, mm);
        mxArray* cm = mxCreateDoubleMatrix(n, 3, mxREAL);
        for (i = 0; i < n; ++i) { int j; for (j = 0; j < 3; ++j) real_data(cm)[(size_t)j * n + i] = (double)ch[3 * i + j]; }
        OUT(1, cm);
    } else if (!strcmp(op, "sweep_papr")) {   /* [hist (n_bins x n_points), PAPR (spp x n_points)] =
                                                 sweep_papr(LINK..., scramble, p_one, streams_per_point, seed, bin_db, n_bins, pool, pool_stride):
                                                 scramble / p_one one entry per point (p_one ignored with a pool); pool = 0/1 payload
                                                 bits (e.g. file_reader's) or [] for the Philox Bernoulli payload; hist counts the
                                                 window PAPR values in bins of bin_db dB, the last bin takes everything above it */
        NEED(N_LINK + 8);
        ofdm_link_params lp;
        ofdm_papr_params pp;
        parse_link(&A(0), &lp);
        memset(&pp, 0, sizeof pp);
        size_t n = mxGetNumberOfElements(A(N_LINK)), i;
        if (!n) fail("ofdm:sweep_papr:points", "need at least one point");
        size_t npool = mxGetNumberOfElements(A(N_LINK + 6));
        if (!npool && mxGetNumberOfElements(A(N_LINK + 1)) != n) fail("ofdm:sweep_papr:p_one", "p_one must have one entry per point");
        int32_t* scr = (int32_t*)hostbuf(n * 4);
        for (i = 0; i < n; ++i) scr[i] = real_data(A(N_LINK))[i] != 0.0;
        pp.n_points = (int32_t)n;
        pp.scramble_host = scr;
        pp.p_one_host = npool ? NULL : real_data(A(N_LINK + 1));
        if (npool) {
            uint32_t* pw = (uint32_t*)hostbuf(OFDM_BIT_WORDS(npool) * 4);
            const double* pb = real_data(A(N_LINK + 6));
            for (i = 0; i < npool; ++i) if (pb[i] != 0.0) pw[i >> 5] |= 1u << (i & 31);
            pp.pool_host = pw;
            pp.pool_bits = (int64_t)npool;
            pp.pool_stride = (int64_t)mxGetScalar(A(N_LINK + 7));
        }
        pp.streams_per_point = (int64_t)mxGetScalar(A(N_LINK + 2));
        pp.rank = 0; pp.world = 1;
        pp.seed = (uint64_t)mxGetScalar(A(N_LINK + 3));
        pp.bin_db = mxGetScalar(A(N_LINK + 4));
        pp.n_bins = (int32_t)mxGetScalar(A(N_LINK + 5));
        size_t spp = (size_t)(pp.streams_per_point > 0 ? pp.streams_per_point : 0), nb = (size_t)(pp.n_bins > 0 ? pp.n_bins : 0);
        int64_t* hh = (int64_t*)hostbuf(n * nb * 8 + 8);
        mxArray* pm = mxCreateDoubleMatrix(spp, n, mxREAL);
        if (sweep_group()) chk_group(ofdm_group_sweep_papr(g_group, &lp, &pp, spp ? real_data(pm) : (double*)hostbuf(8), hh), op);
        else {
            double* pd = (double*)devbuf(n * spp * 8 + 8);
            int64_t* hd = (int64_t*)devbuf(n * nb * 8 + 8);
            chk(ofdm_memset(g_ctx, pd, 0, n * spp * 8), "memset");
            chk(ofdm_memset(g_ctx, hd, 0, n * nb * 8), "memset");
            chk(ofdm_sweep_papr(g_ctx, &lp, &pp, pd, hd), op);
            chk(ofdm_d2h(g_ctx, hh, hd, n * nb * 8), "d2h");
            chk(ofdm_d2h(g_ctx, real_data(pm), pd, n * spp * 8), "d2h");
        }
        mxArray* hm = mxCreateDoubleMatrix(nb, n, mxREAL);
        for (i = 0; i < n * nb; ++i) real_data(hm)[i] = (double)hh[i];
        OUT(0, hm);
        OUT(1, pm);
    } else if (!strcmp(op, "sweep_part2")) {   /* [NMSE (4 x n_points), BER (4 x n_points), per_run (mc_runs x 4*n_points), counts (12 x n_points),
                                                   runs (2 x n_points)] = sweep_part2(Nfft, T_Guard, N_carrier, N_symb, SpF, Constellation,
                                                   pilots, offsets, Ldict, pattern, bits, profile, fs, SNR, monteCarloRuns, seed, near_eps, tie_eps):
                                                   offsets = [] -> pilots is a vector of combs (pilots 1:comb:N_carrier, Ldict ceil(Nfft/comb));
                                                   else pilots are the concatenated 1-based pilot vectors of the points, offsets (n_points + 1,
                                                   from 0) delimit them and Ldict defaults to Nfft.  Ldict = [] takes the defaults.  pattern: the
                                                   two pilot values (pilot q carries pattern(mod(q-1,2)+1)).  bits: 0/1 payload. */
        NEED(18);
        ofdm_link_params lp;
        ofdm_part2_params pp;
        char prof[8];
        size_t i, P, n_comb = mxGetNumberOfElements(A(6)), n_off = mxGetNumberOfElements(A(7));
        int e;
        memset(&lp, 0, sizeof lp);
        memset(&pp, 0, sizeof pp);
        lp.Nfft = (int32_t)mxGetScalar(A(0)); lp.Tg = (int32_t)mxGetScalar(A(1)); lp.N_carrier = (int32_t)mxGetScalar(A(2));
        lp.S = (int32_t)mxGetScalar(A(3)); lp.SpF = (int32_t)mxGetScalar(A(4));
        lp.constellation = constellation_id(A(5));
        const double* pil = real_data(A(6));
        int32_t* off; int32_t* car; int32_t* ld;
        if (n_off == 0) {                                               /* combs (`Task5_part2.m:50-55`) */
            size_t tot = 0;
            P = n_comb;
            if (!P) fail("ofdm:sweep_part2:pilots", "need at least one comb");
            for (i = 0; i < P; ++i) {
                if (pil[i] < 1) fail("ofdm:sweep_part2:pilots", "combs must be >= 1");
                tot += (size_t)((lp.N_carrier + (int)pil[i] - 1) / (int)pil[i]);
            }
            off = (int32_t*)hostbuf((P + 1) * 4); car = (int32_t*)hostbuf(tot * 4 + 4); ld = (int32_t*)hostbuf(P * 4);
            for (i = 0; i < P; ++i) {
                int comb = (int)pil[i], c;
                off[i + 1] = off[i];
                for (c = 1; c <= lp.N_carrier; c += comb) car[off[i + 1]++] = c;
                ld[i] = (lp.Nfft + comb - 1) / comb;                    /* F(:,1:ceil(Nfft/comb)), `:183-185` */
            }
        } else {                                                        /* explicit pilot vectors (random masks, `:57-65`) */
            const double* po = real_data(A(7));
            P = n_off - 1;
            if (!P) fail("ofdm:sweep_part2:pilots", "offsets must have n_points + 1 entries");
            off = (int32_t*)hostbuf((P + 1) * 4); car = (int32_t*)hostbuf(n_comb * 4 + 4); ld = (int32_t*)hostbuf(P * 4);
            for (i = 0; i <= P; ++i) {
                off[i] = (int32_t)llround(po[i]);
                if (off[i] < 0 || (size_t)off[i] > n_comb) fail("ofdm:sweep_part2:pilots", "offsets must lie in 0..numel(pilots)");
            }
            for (i = 0; i < n_comb; ++i) car[i] = (int32_t)llround(pil[i]);
            for (i = 0; i < P; ++i) ld[i] = lp.Nfft;
        }
        if (mxGetNumberOfElements(A(8))) {
            if (mxGetNumberOfElements(A(8)) != P) fail("ofdm:sweep_part2:ldict", "Ldict must have one entry per point");
            for (i = 0; i < P; ++i) ld[i] = (int32_t)llround(real_data(A(8))[i]);
        }
        if (mxGetNumberOfElements(A(9)) != 2) fail("ofdm:sweep_part2:pattern", "the pilot pattern must have two values");
        size_t nbits = mxGetNumberOfElements(A(10));
        uint32_t* words = (uint32_t*)hostbuf(OFDM_BIT_WORDS(nbits) * 4 + 4);
        for (i = 0; i < nbits; ++i) if (real_data(A(10))[i] != 0.0) words[i >> 5] |= 1u << (i & 31);
        if (!mxIsChar(A(11)) || mxGetString(A(11), prof, sizeof prof)) fail("ofdm:sweep_part2:profile", "profile must be 'EPA', 'EVA' or 'ETU'");
        pp.profile = !strcmp(prof, "EPA") ? 0 : !strcmp(prof, "EVA") ? 1 : !strcmp(prof, "ETU") ? 2 : -1;
        if (pp.profile < 0) fail("ofdm:sweep_part2:profile", "profile must be 'EPA', 'EVA' or 'ETU'");
        pp.n_points = (int32_t)P;
        pp.pilot_offsets_host = off; pp.pilot_carriers_host = car; pp.ldict_host = ld;
        pp.pilot_pattern_host = to_cdoubles(A(9), 2);
        pp.payload_host = words; pp.payload_bits = (int64_t)nbits;
        pp.fs_hz = mxGetScalar(A(12)); pp.snr_db = mxGetScalar(A(13));
        pp.mc_runs = (int64_t)mxGetScalar(A(14));
        pp.rank = 0; pp.world = 1;
        pp.seed = (uint64_t)mxGetScalar(A(15));
        pp.near_eps = mxGetScalar(A(16)); pp.tie_eps = mxGetScalar(A(17));
        size_t R = (size_t)(pp.mc_runs > 0 ? pp.mc_runs : 0), cells = P * 4 * R;
        double* mh = (double*)hostbuf(cells * 8 + 8);
        int64_t* ch = (int64_t*)hostbuf(P * 96);
        int64_t* rh = (int64_t*)hostbuf(P * 16);
        if (sweep_group()) chk_group(ofdm_group_sweep_part2(g_group, &lp, &pp, mh, ch, rh), op);
        else {
            double* md = (double*)devbuf(cells * 8 + 8);
            int64_t* cd = (int64_t*)devbuf(P * 96);
            int64_t* rd = (int64_t*)devbuf(P * 16);
            chk(ofdm_memset(g_ctx, md, 0, cells * 8), "memset");
            chk(ofdm_memset(g_ctx, cd, 0, P * 96), "memset");
            chk(ofdm_memset(g_ctx, rd, 0, P * 16), "memset");
            chk(ofdm_sweep_part2(g_ctx, &lp, &pp, md, cd, rd), op);
            chk(ofdm_d2h(g_ctx, mh, md, cells * 8), "d2h");
            chk(ofdm_d2h(g_ctx, ch, cd, P * 96), "d2h");
            chk(ofdm_d2h(g_ctx, rh, rd, P * 16), "d2h");
        }
        mxArray* nm = mxCreateDoubleMatrix(4, P, mxREAL);              /* `Task5_part2.m:305-314`: estimators x points */
        mxArray* bm = mxCreateDoubleMatrix(4, P, mxREAL);
        for (i = 0; i < P; ++i)
            for (e = 0; e < 4; ++e) {
                double s = 0; size_t r;
                for (r = 0; r < R; ++r) s += mh[(i * 4 + e) * R + r];
                real_data(nm)[i * 4 + e] = s / (double)R;
                real_data(bm)[i * 4 + e] = (double)ch[i * 12 + 3 * e] / (double)ch[i * 12 + 3 * e + 1];
            }
        OUT(0, nm);
        OUT(1, bm);
        mxArray* pm = mxCreateDoubleMatrix(R, 4 * P, mxREAL);          /* reshape(per_run, mc_runs, 4, n_points) in MATLAB */
        memcpy(real_data(pm), mh, cells * 8);
        OUT(2, pm);
        mxArray* cm = mxCreateDoubleMatrix(12, P, mxREAL);             /* reshape(counts, 3, 4, n_points): {errors, bits, near} */
        for (i = 0; i < 12 * P; ++i) real_data(cm)[i] = (double)ch[i];
        OUT(3, cm);
        mxArray* rm = mxCreateDoubleMatrix(2, P, mxREAL);              /* {runs, OMP runs with a near-tie} */
        for (i = 0; i < 2 * P; ++i) real_data(rm)[i] = (double)rh[i];
        OUT(4, rm);
    } else {
        fail("ofdm:arg:op", "unknown operation");
    }
    release_all();
}
