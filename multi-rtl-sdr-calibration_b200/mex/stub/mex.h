/* mex.h - minimal stand-in for the MATLAB/Octave MEX API, enough to compile mex/gsmcal_mex.c and drive its gateways from a C
 * test harness.  NOT a MATLAB replacement.  Default: split complex (Octave, pre-R2018a MATLAB: mxGetPr/mxGetPi); with
 * -DMX_HAS_INTERLEAVED_COMPLEX=1: the -R2018a flavour (mxGetComplexDoubles / mxGetDoubles, complex data interleaved in `re`). */
#ifndef GSMCAL_STUB_MEX_H
#define GSMCAL_STUB_MEX_H
#include <math.h>
#include <stdarg.h>
#include <stddef.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

typedef enum { mxREAL = 0, mxCOMPLEX = 1 } mxComplexity;
typedef enum { mxDOUBLE_CLASS = 6, mxUINT8_CLASS = 9, mxLOGICAL_CLASS = 3, mxSTRUCT_CLASS = 2 } mxClassID;
typedef struct mxArray_tag {
    mxClassID cls; int is_complex; size_t ndim; size_t dims[3];
    void *re; void *im;
    int nfields; const char **fnames;     /* struct arrays: re holds nfields mxArray* per element */
} mxArray;
typedef int bool_t_;

static void mexErrMsgIdAndTxt(const char *id, const char *fmt, ...) {
    va_list ap; va_start(ap, fmt); fprintf(stderr, "MEX error %s: ", id); vfprintf(stderr, fmt, ap); fprintf(stderr, "\n"); va_end(ap);
    exit(3);
}
static int mexPrintf(const char *fmt, ...) { va_list ap; va_start(ap, fmt); int n = vprintf(fmt, ap); va_end(ap); return n; }
static void (*mex_at_exit_fn)(void) = NULL;
static int mexAtExit(void (*fn)(void)) { mex_at_exit_fn = fn; return 0; }
static void *mxMalloc(size_t n) { return malloc(n ? n : 1); }
static void mxFree(void *p) { free(p); }
static size_t mxGetNumberOfElements(const mxArray *a) { size_t n = 1; for (size_t i = 0; i < a->ndim; ++i) n *= a->dims[i]; return n; }
static size_t mxGetM(const mxArray *a) { return a->dims[0]; }
static size_t mxGetN(const mxArray *a) { size_t n = 1; for (size_t i = 1; i < a->ndim; ++i) n *= a->dims[i]; return n; }
static int mxIsDouble(const mxArray *a) { return a->cls == mxDOUBLE_CLASS; }
static int mxIsUint8(const mxArray *a) { return a->cls == mxUINT8_CLASS; }
static int mxIsComplex(const mxArray *a) { return a->is_complex; }
static double *mxGetPr(const mxArray *a) { return (double *)a->re; }
static double *mxGetPi(const mxArray *a) { return (double *)a->im; }
static void *mxGetData(const mxArray *a) { return a->re; }
static double mxGetScalar(const mxArray *a) { return a->cls == mxDOUBLE_CLASS ? ((double *)a->re)[0] : (double)((unsigned char *)a->re)[0]; }
static double mxGetNaN(void) { return NAN; }
static mxArray *mxCreateNumericArray(size_t ndim, const size_t *dims, mxClassID cls, mxComplexity c) {
    mxArray *a = (mxArray *)calloc(1, sizeof(mxArray));
    a->cls = cls; a->is_complex = (c == mxCOMPLEX); a->ndim = ndim;
    size_t n = 1; for (size_t i = 0; i < ndim; ++i) { a->dims[i] = dims[i]; n *= dims[i]; }
    size_t es = (cls == mxDOUBLE_CLASS) ? 8 : 1;
#if defined(MX_HAS_INTERLEAVED_COMPLEX) && MX_HAS_INTERLEAVED_COMPLEX
    a->re = calloc((n ? n : 1) * (a->is_complex ? 2 : 1), es); a->im = NULL;
#else
    a->re = calloc(n ? n : 1, es); a->im = a->is_complex ? calloc(n ? n : 1, es) : NULL;
#endif
    return a;
}
#if defined(MX_HAS_INTERLEAVED_COMPLEX) && MX_HAS_INTERLEAVED_COMPLEX
typedef struct { double real, imag; } mxComplexDouble;
static mxComplexDouble *mxGetComplexDoubles(const mxArray *a) { return (mxComplexDouble *)a->re; }
static double *mxGetDoubles(const mxArray *a) { return (double *)a->re; }
#endif
static mxArray *mxCreateDoubleMatrix(size_t m, size_t n, mxComplexity c) { size_t d[2] = {m, n}; return mxCreateNumericArray(2, d, mxDOUBLE_CLASS, c); }
static mxArray *mxCreateDoubleScalar(double v) { mxArray *a = mxCreateDoubleMatrix(1, 1, mxREAL); ((double *)a->re)[0] = v; return a; }
static mxArray *mxCreateLogicalScalar(int v) { size_t d[2] = {1, 1}; mxArray *a = mxCreateNumericArray(2, d, mxLOGICAL_CLASS, mxREAL); ((unsigned char *)a->re)[0] = v ? 1 : 0; return a; }
static mxArray *mxCreateStructMatrix(size_t m, size_t n, int nfields, const char **fieldnames) {
    mxArray *a = (mxArray *)calloc(1, sizeof(mxArray));
    a->cls = mxSTRUCT_CLASS; a->ndim = 2; a->dims[0] = m; a->dims[1] = n; a->nfields = nfields;
    a->fnames = (const char **)calloc((size_t)nfields, sizeof(char *));
    for (int f = 0; f < nfields; ++f) a->fnames[f] = fieldnames[f];
    a->re = calloc((m * n ? m * n : 1) * (size_t)nfields, sizeof(mxArray *));
    return a;
}
static int mxIsStruct(const mxArray *a) { return a->cls == mxSTRUCT_CLASS; }
static int mx_field_(const mxArray *a, const char *name) { for (int f = 0; f < a->nfields; ++f) if (!strcmp(a->fnames[f], name)) return f; return -1; }
static void mxSetField(mxArray *a, size_t i, const char *name, mxArray *v) { int f = mx_field_(a, name); if (f >= 0) ((mxArray **)a->re)[i * a->nfields + f] = v; }
static mxArray *mxGetField(const mxArray *a, size_t i, const char *name) { int f = mx_field_(a, name); return f < 0 ? NULL : ((mxArray **)a->re)[i * a->nfields + f]; }
static void mxDestroyArray(mxArray *a) { if (a) { free(a->re); free(a->im); free(a); } }

void mexFunction(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[]);
#endif
