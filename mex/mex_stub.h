/* mex_stub.h -- the handful of MATLAB MEX declarations wofdm_mex.cpp uses, so the gateway can be
 * compile-checked (g++ -fsyntax-only -DWOFDM_MEX_STUB) where MATLAB is not installed.  With MATLAB,
 * build with `mex -I../include wofdm_mex.cpp -L../w-ofdm-optimization_b200 -lwofdm` and this file is unused. */
#ifndef WOFDM_MEX_STUB_H_
#define WOFDM_MEX_STUB_H_
#include <stddef.h>
typedef struct mxArray_tag mxArray;
typedef size_t mwSize;
typedef enum { mxREAL = 0, mxCOMPLEX = 1 } mxComplexity;
typedef enum { mxDOUBLE_CLASS = 6 } mxClassID;
extern "C" {
double* mxGetPr(const mxArray*);
double* mxGetPi(const mxArray*);
double mxGetScalar(const mxArray*);
size_t mxGetM(const mxArray*);
size_t mxGetN(const mxArray*);
size_t mxGetNumberOfElements(const mxArray*);
bool mxIsChar(const mxArray*);
bool mxIsCell(const mxArray*);
mxArray* mxGetCell(const mxArray*, size_t);
bool mxIsComplex(const mxArray*);
int mxGetString(const mxArray*, char*, mwSize);
mxArray* mxCreateDoubleMatrix(mwSize, mwSize, mxComplexity);
mxArray* mxCreateDoubleScalar(double);
mxArray* mxCreateNumericArray(mwSize, const mwSize*, mxClassID, mxComplexity);
void mexErrMsgIdAndTxt(const char*, const char*, ...);
int mexAtExit(void (*)(void));
}
#endif
