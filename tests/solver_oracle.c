/*
 * solver_oracle.c -- CPU oracle of the Nesterov, AdaGrad, RMSProp and AdaDelta updates (test infrastructure).
 *
 * The sync half (on_start all-gather, 1/N scale, ordered reduce-scatter) and SGD stay in oracle/sync_oracle.c;
 * this file restates SGDSolver::ApplyUpdate (sgd_solver.cpp:102-116) for the other solvers of the reference:
 * Regularize (sgd_solver.cpp:145-172), the CPU case of <type>_solver.cpp ComputeUpdateValue, Blob::Update
 * (blob.cpp:162-179).  Paths are relative to caffe-public/ of the reference.
 *
 * Build: cc -O2 -ffp-contract=off -fno-fast-math -fPIC -shared -lm.  Every fp32 operation below is one
 * rounding, in the netlib-style BLAS order of mkl_alternate.hpp / math_functions.cpp:
 *   caffe_cpu_axpby(n, a, x, b, y)   y = b*y; y = a*x + y       (cblas_sscal then cblas_saxpy)
 *   caffe_add(n, a, b, y)            y = a + b
 *   caffe_add_scalar(n, d, y)        y = y + d
 *   caffe_div(n, a, b, y)            y = a / b
 *   caffe_mul(n, a, b, y)            y = a * b
 *   caffe_cpu_scale(n, a, x, y)      y = a * x
 *   caffe_powx(n, x, 2, y)           y = x * x        (glibc powf(x, 2) == x*x for every float)
 *   caffe_powx(n, x, 0.5, y)         y = sqrtf(x)     (correctly rounded; glibc powf(x, 0.5) differs by 1 ulp on
 *                                                      ~0.06 % of inputs, DESIGN.md §7)
 */
#include <math.h>
#include <stdint.h>

enum { SOLVER_SGD = 0, SOLVER_NESTEROV = 1, SOLVER_ADAGRAD = 2, SOLVER_RMSPROP = 3, SOLVER_ADADELTA = 4 };

/* One element: g = diff, w = data, h = history_[k], h2 = history_[n + k] (AdaDelta). */
static void update_element(int type, float* gp, float* wp, float* hp, float* h2p, float local_rate, float local_decay,
                           int l1, float momentum, float delta, float rms_decay) {
  float g = *gp, w = *wp, h = *hp, h2 = h2p ? *h2p : 0.f, u, t;
  /* Regularize sgd_solver.cpp:155-168: caffe_axpy(local_decay, data or sign(data), diff) */
  if (local_decay != 0.f) {
    float x = l1 ? (float)((0.f < w) - (w < 0.f)) : w;
    t = local_decay * x;
    g = t + g;
  }
  switch (type) {
    case SOLVER_NESTEROV: {
      const float one_plus_m = 1.0f + momentum, neg_m = -momentum; /* Dtype(1) + momentum, -momentum */
      u = h;                                       /* nesterov_solver.cpp:23-25 caffe_copy(history -> update) */
      h = momentum * h;                            /* :28-30 caffe_cpu_axpby(local_rate, diff, momentum, history) */
      t = local_rate * g;
      h = t + h;
      u = neg_m * u;                               /* :33-35 caffe_cpu_axpby(1 + m, history, -m, update) */
      t = one_plus_m * h;
      u = t + u;
      g = u;                                       /* :38-40 caffe_copy(update -> diff) */
      break;
    }
    case SOLVER_ADAGRAD:
    case SOLVER_RMSPROP:
      u = g * g;                                   /* adagrad :23-25, rmsprop :26-28 caffe_powx(diff, 2) */
      if (type == SOLVER_ADAGRAD) {
        h = u + h;                                 /* adagrad :28-31 caffe_add(update, history, history) */
      } else {
        const float one_minus = 1.0f - rms_decay;  /* rmsprop :31-33 axpby(Dtype(1-rms_decay), update, rms_decay, h) */
        h = rms_decay * h;
        t = one_minus * u;
        h = t + h;
      }
      u = sqrtf(h);                                /* adagrad :34-36, rmsprop :36-38 caffe_powx(history, 0.5) */
      u = u + delta;                               /* adagrad :38-39, rmsprop :40-41 caffe_add_scalar(delta) */
      u = g / u;                                   /* adagrad :41-44, rmsprop :43-45 caffe_div(diff, update) */
      g = 0.0f * g;                                /* adagrad :47-49, rmsprop :48-50 axpby(local_rate, update, 0, diff) */
      t = local_rate * u;
      g = t + g;
      break;
    case SOLVER_ADADELTA: {
      const float one_minus = 1.0f - momentum;     /* Dtype(1) - momentum */
      u = g * g;                                   /* adadelta_solver.cpp:36-38 caffe_powx(diff, 2) */
      h = momentum * h;                            /* :41-43 axpby(1 - m, update, m, history) */
      t = one_minus * u;
      h = t + h;
      u = delta + h2;                              /* :46-52 caffe_set(temp, delta); caffe_add(temp, h2, update) */
      t = delta + h;                               /* :54-57 caffe_add(temp, history, temp) */
      u = u / t;                                   /* :60-63 caffe_div(update, temp, update) */
      u = sqrtf(u);                                /* :66-68 caffe_powx(update, 0.5) */
      g = g * u;                                   /* :71-74 caffe_mul(diff, update, diff) */
      u = g * g;                                   /* :77-79 caffe_powx(diff, 2) */
      h2 = momentum * h2;                          /* :82-84 axpby(1 - m, update, m, history[n + i]) */
      t = one_minus * u;
      h2 = t + h2;
      g = local_rate * g;                          /* :87-89 caffe_cpu_scale(local_rate, diff, diff) */
      break;
    }
    default: /* SGD, sgd_solver.cpp:213-229 */
      h = momentum * h;
      t = local_rate * g;
      h = t + h;
      g = h;
  }
  t = -1.0f * g; /* blob.cpp:162-179 caffe_axpy(-1, diff, data) */
  w = t + w;
  *gp = g;
  *wp = w;
  *hp = h;
  if (h2p) *h2p = h2;
}

/* ApplyUpdate over elements [begin, end) of a flat layout of nblobs blobs; hist2 may be NULL unless AdaDelta. */
void cos_solver_oracle_apply_update(uint64_t begin, uint64_t end, float* data, float* diff, float* hist, float* hist2,
                                    int nblobs, const int64_t* counts, const float* lr_mult, const float* decay_mult,
                                    float rate, float momentum, float weight_decay, int l1, int type, float delta,
                                    float rms_decay) {
  uint64_t blob_begin = 0;
  for (int k = 0; k < nblobs; ++k) {
    const uint64_t blob_end = blob_begin + (uint64_t)counts[k];
    const uint64_t lo = blob_begin > begin ? blob_begin : begin;
    const uint64_t hi = blob_end < end ? blob_end : end;
    const float local_decay = weight_decay * decay_mult[k]; /* sgd_solver.cpp:151 */
    const float local_rate = rate * lr_mult[k];             /* <type>_solver.cpp: rate * net_params_lr[param_id] */
    for (uint64_t i = lo; i < hi; ++i)
      update_element(type, diff + i, data + i, hist + i, type == SOLVER_ADADELTA ? hist2 + i : 0, local_rate,
                     local_decay, l1, momentum, delta, rms_decay);
    blob_begin = blob_end;
  }
}
