/* nnsp_model.h -- host-side model object: a reference `NeuralNetClass` table
 * (evb/src/def_nn*.c) read into a self-contained, canonical form.
 *
 * Canonical weight layout (what every GPU layout is derived from):
 *   fc   layer : W[row][col], row-major int8, rows = size_layer[i+1], cols = size_layer[i]
 *   lstm layer : W[gate*H + unit][col] and Wrec[gate*H + unit][H], gate order i, j(g), f, o
 *                (python/nnsp_pack/c_weight_man.py:61-92, ns-nnsp/src/lstm.c:54-104);
 *                bias[gate*H + unit]
 * The ARM 4-row interleave of the table files (c_weight_man.py:5-47, affine.c:74-184) is
 * undone at load time and re-applied by nnsp_b200_model_to_blob, so tables round-trip.
 */
#ifndef NNSP_MODEL_H
#define NNSP_MODEL_H
#include <stddef.h>
#include <stdint.h>
#include "nnsp_b200.h"
#ifdef __cplusplus
extern "C" {
#endif

enum { NNSP_LAYER_FC = 0, NNSP_LAYER_LSTM = 1 };
enum { NNSP_ACT_RELU6 = 0, NNSP_ACT_TANH = 1, NNSP_ACT_SIGMOID = 2, NNSP_ACT_LINEAR = 3 };

typedef struct {
    int      type;          /* NNSP_LAYER_* */
    int      act;           /* NNSP_ACT_*  (ignored by lstm layers, lstm.c:65-104) */
    int      rows, cols;    /* units out, units in */
    int      qk, qi, qb;    /* qbit_kernel / qbit_input / qbit_bias */
    int      qi_next;       /* qbit_input of the next layer (= qbit_input_rec, neural_nets.c:108) */
    int      acc32;         /* 1: wrapping 32-bit accumulator semantics (affine_acc32b.c) */
    int8_t  *w;             /* canonical [nrows_total][cols]; nrows_total = rows (fc) or 4*rows (lstm) */
    int8_t  *wrec;          /* lstm only: canonical [4*rows][rows] */
    int16_t *bias;          /* [nrows_total] */
} nnsp_layer;

struct nnsp_b200_model {
    int        nn_id;
    int        numlayers;
    int16_t    size_layer[NNSP_B200_MAX_LAYERS + 1];
    int32_t    mean[NNSP_B200_NMEL];
    int32_t    stdR[NNSP_B200_NMEL];
    nnsp_layer layer[NNSP_B200_MAX_LAYERS];
};

/* ARM 4-row interleave <-> canonical row-major, for one `rows x cols` matrix laid out by
 * c_matrix_man (4-row blocks, then a 1..3-row remainder block; 2x2 transposed tiles; odd
 * last column stored column-wise). Both return the number of bytes consumed/produced. */
size_t nnsp_deinterleave_arm(const int8_t *src, int rows, int cols, int8_t *dst_rowmajor);
size_t nnsp_interleave_arm(const int8_t *src_rowmajor, int rows, int cols, int8_t *dst);

void nnsp_set_error(const char *fmt, ...);

/* nnsp_cascade.cu: NNSP_B200_ERR_ARG unless all n records may be imported into handle c (nnsp_b200_cascade_import_streams) */
int nnsp_cascade_check_records(const nnsp_b200_cascade *c, const void *records, int n);

#ifdef __cplusplus
}
#endif
#endif
