/* ba_schur_blocks.h — block-sparse assembly and band(+arrow) Cholesky of the reduced camera
 * system for the CPU oracle (TEST INFRASTRUCTURE; included by ba_oracle.c only).
 *
 * What it restates: Ceres SPARSE_SCHUR, the solver the reference selects for 50 < F <= 1000
 * images (bundle_adjustment.cc:276-286): SchurEliminator writes S as a BLOCK-SPARSE matrix whose
 * blocks are the image pairs that co-observe a point, and a sparse Cholesky (CHOLMOD) factors
 * it.  For a video the co-visible pairs form a band, whose fill stays inside the band.
 * Round 1 assembled a dense (6F+3)^2 S with up to 16 private dense copies and a dense
 * Cholesky: that neither scales with threads nor resembles SPARSE_SCHUR.  Here:
 *   - pattern: image pairs (a <= b) sharing a point -> block ids (once per problem)
 *   - per THREAD a private array of block values (F * (span + 1) * 36 doubles for a video:
 *     cache resident), merged by a parallel sum — no atomics, no dense copies
 *   - banded: Cholesky in band storage, O(n bw^2); the shared camera's 3 slots are an arrow
 *   - not banded (span > F / 2): scattered into the dense S and factored by chol_lower()
 * Single shared camera only (the pipeline's single_camera = 1); ba_oracle.c keeps the
 * general dense path for C > 1.
 */
#ifndef PSFM_ORACLE_BA_SCHUR_BLOCKS_H
#define PSFM_ORACLE_BA_SCHUR_BLOCKS_H

typedef struct {
  int ready;
  int nblk, span;        /* number of image-pair blocks, max (b - a) */
  int* blk_of;           /* [F * F] block id of pair (a, b), a <= b; -1 when absent */
  int* blk_a; int* blk_b;
  size_t stride;         /* doubles per thread: nblk * 36 + F * 18 + 9, padded */
  double* acc;           /* [nthreads][stride] */
  double* sum;           /* [stride] merged */
  double* AB;            /* band storage [6F][bw + 1] */
  double* AR;            /* arrow rows [3][6F] */
} sblocks_t;

static void sblocks_free(sblocks_t* s) {
  free(s->blk_of); free(s->blk_a); free(s->blk_b); free(s->acc); free(s->sum); free(s->AB); free(s->AR);
  memset(s, 0, sizeof(*s));
}

/* image pairs (a <= b) that share a point */
static int sblocks_pattern(sblocks_t* s, int F, int P, const int* pt_ptr, const int* pt_obs, const int* obs_image,
                           int nthreads) {
  if ((size_t)F * F > ((size_t)1 << 28)) return 1;
  s->blk_of = (int*)malloc(sizeof(int) * (size_t)F * F);
  if (!s->blk_of) return 1;
  for (size_t k = 0; k < (size_t)F * F; ++k) s->blk_of[k] = -1;
  for (int p = 0; p < P; ++p) {
    const int b = pt_ptr[p], e = pt_ptr[p + 1];
    for (int i = b; i < e; ++i) {
      const int ia = obs_image[pt_obs[i]];
      for (int j = i; j < e; ++j) {
        const int ib = obs_image[pt_obs[j]];
        const int lo = ia < ib ? ia : ib, hi = ia < ib ? ib : ia;
        s->blk_of[(size_t)lo * F + hi] = 0;
      }
    }
  }
  int n = 0, span = 0;
  for (int a = 0; a < F; ++a)
    for (int b = a; b < F; ++b)
      if (s->blk_of[(size_t)a * F + b] == 0) { ++n; if (b - a > span) span = b - a; }
  s->blk_a = (int*)malloc(sizeof(int) * (size_t)(n + 1));
  s->blk_b = (int*)malloc(sizeof(int) * (size_t)(n + 1));
  n = 0;
  for (int a = 0; a < F; ++a)
    for (int b = a; b < F; ++b)
      if (s->blk_of[(size_t)a * F + b] == 0) { s->blk_of[(size_t)a * F + b] = n; s->blk_a[n] = a; s->blk_b[n] = b; ++n; }
  s->nblk = n; s->span = span;
  s->stride = ((size_t)n * 36 + (size_t)F * 18 + 9 + 7) & ~(size_t)7;
  s->acc = (double*)malloc(sizeof(double) * s->stride * (size_t)nthreads);
  s->sum = (double*)malloc(sizeof(double) * s->stride);
  if (!s->blk_a || !s->blk_b || !s->acc || !s->sum) return 1;
  s->ready = 1;
  return 0;
}

/* S = F'F - sum_p (F'E) Hinv (E'F) in block form.  Jc [M][2][6], Jp [M][2][3], Jk [M][2][3]
   (column scaled), Hinv [P][9].  Result in s->sum: blocks (a <= b; (a, a) full symmetric),
   then the pose x intrinsics blocks [F][6][3], then the intrinsics block [3][3]. */
static void sblocks_assemble(sblocks_t* s, int F, int P, const int* pt_ptr, const int* pt_obs, const int* obs_image,
                             const double* Jc, const double* Jp, const double* Jk, const double* Hinv, int nthreads) {
  const size_t st = s->stride;
#pragma omp parallel num_threads(nthreads)
  {
#ifdef _OPENMP
    const int th = omp_get_thread_num();
#else
    const int th = 0;
#endif
    double* A = s->acc + st * (size_t)th;
    double* Acol = A + (size_t)s->nblk * 36;
    double* Akk = Acol + (size_t)F * 18;
    memset(A, 0, sizeof(double) * st);
    int wcap = 64;
    double* W = (double*)malloc(sizeof(double) * 18 * (size_t)wcap);
    double* WH = (double*)malloc(sizeof(double) * 18 * (size_t)wcap);
    int* im = (int*)malloc(sizeof(int) * (size_t)wcap);
#pragma omp for schedule(dynamic, 256)
    for (int p = 0; p < P; ++p) {
      const int b = pt_ptr[p], L = pt_ptr[p + 1] - b;
      if (L == 0) continue;
      if (L > wcap) {
        wcap = L;
        W = (double*)realloc(W, sizeof(double) * 18 * (size_t)wcap);
        WH = (double*)realloc(WH, sizeof(double) * 18 * (size_t)wcap);
        im = (int*)realloc(im, sizeof(int) * (size_t)wcap);
      }
      const double* Hi = Hinv + 9 * (size_t)p;
      double wks[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};      /* sum_j Wk_j  (3 x 3) */
      for (int e = 0; e < L; ++e) {
        const int i = pt_obs[b + e];
        const double* jc = Jc + 12 * (size_t)i;
        const double* jp = Jp + 6 * (size_t)i;
        const double* jk = Jk + 6 * (size_t)i;
        const int img = obs_image[i];
        im[e] = img;
        double* w = W + 18 * (size_t)e;
        double* wh = WH + 18 * (size_t)e;
        for (int a = 0; a < 6; ++a)
          for (int k = 0; k < 3; ++k) w[3 * a + k] = jc[a] * jp[k] + jc[6 + a] * jp[3 + k];
        for (int a = 0; a < 6; ++a)
          for (int k = 0; k < 3; ++k) wh[3 * a + k] = w[3 * a] * Hi[k] + w[3 * a + 1] * Hi[3 + k] + w[3 * a + 2] * Hi[6 + k];
        for (int a = 0; a < 3; ++a)
          for (int k = 0; k < 3; ++k) wks[3 * a + k] += jk[a] * jp[k] + jk[3 + a] * jp[3 + k];
        /* F'F */
        double* D = A + 36 * (size_t)s->blk_of[(size_t)img * F + img];
        for (int a = 0; a < 6; ++a)
          for (int k = 0; k < 6; ++k) D[6 * a + k] += jc[a] * jc[k] + jc[6 + a] * jc[6 + k];
        double* Cc = Acol + 18 * (size_t)img;
        for (int a = 0; a < 6; ++a)
          for (int k = 0; k < 3; ++k) Cc[3 * a + k] += jc[a] * jk[k] + jc[6 + a] * jk[3 + k];
        for (int a = 0; a < 3; ++a)
          for (int k = 0; k < 3; ++k) Akk[3 * a + k] += jk[a] * jk[k] + jk[3 + a] * jk[3 + k];
      }
      /* - (W Hinv) W' over the ordered pairs with image_i <= image_j */
      for (int ei = 0; ei < L; ++ei) {
        const double* whi = WH + 18 * (size_t)ei;
        for (int ej = 0; ej < L; ++ej) {
          if (im[ei] > im[ej]) continue;
          const double* wj = W + 18 * (size_t)ej;
          double* D = A + 36 * (size_t)s->blk_of[(size_t)im[ei] * F + im[ej]];
          for (int a = 0; a < 6; ++a)
            for (int k = 0; k < 6; ++k)
              D[6 * a + k] -= whi[3 * a] * wj[3 * k] + whi[3 * a + 1] * wj[3 * k + 1] + whi[3 * a + 2] * wj[3 * k + 2];
        }
        /* pose x intrinsics: - (W_i Hinv) (sum_j Wk_j)' */
        double* Cc = Acol + 18 * (size_t)im[ei];
        for (int a = 0; a < 6; ++a)
          for (int k = 0; k < 3; ++k)
            Cc[3 * a + k] -= whi[3 * a] * wks[3 * k] + whi[3 * a + 1] * wks[3 * k + 1] + whi[3 * a + 2] * wks[3 * k + 2];
      }
      /* intrinsics: - (sum Wk) Hinv (sum Wk)' */
      double wkh[9];
      for (int a = 0; a < 3; ++a)
        for (int k = 0; k < 3; ++k) wkh[3 * a + k] = wks[3 * a] * Hi[k] + wks[3 * a + 1] * Hi[3 + k] + wks[3 * a + 2] * Hi[6 + k];
      for (int a = 0; a < 3; ++a)
        for (int k = 0; k < 3; ++k)
          Akk[3 * a + k] -= wkh[3 * a] * wks[3 * k] + wkh[3 * a + 1] * wks[3 * k + 1] + wkh[3 * a + 2] * wks[3 * k + 2];
    }
    free(W); free(WH); free(im);
  }
#pragma omp parallel for schedule(static) num_threads(nthreads)
  for (long long k = 0; k < (long long)st; ++k) {
    double v = 0.0;
    for (int th = 0; th < nthreads; ++th) v += s->acc[st * (size_t)th + k];
    s->sum[k] = v;
  }
}

/* entry (i, j) of the final system: S + D^2 on active slots, identity on inactive ones */
static inline double sblocks_fix(double v, int i, int j, const unsigned char* active, const double* D) {
  if (!active[i] || !active[j]) return (i == j) ? 1.0 : 0.0;
  return (i == j) ? v + D[i] * D[i] : v;
}

/* scatter the merged blocks into the dense symmetric S [NS][NS] (NS = 6F + 3) */
static void sblocks_to_dense(const sblocks_t* s, int F, const unsigned char* active, const double* Dc, double* S) {
  const int NS = 6 * F + 3;
  memset(S, 0, sizeof(double) * (size_t)NS * NS);
  for (int k = 0; k < s->nblk; ++k) {
    const int a = s->blk_a[k], b = s->blk_b[k];
    const double* B = s->sum + 36 * (size_t)k;
    for (int r = 0; r < 6; ++r)
      for (int c = 0; c < 6; ++c) {
        S[(size_t)(6 * a + r) * NS + 6 * b + c] = B[6 * r + c];
        S[(size_t)(6 * b + c) * NS + 6 * a + r] = B[6 * r + c];
      }
  }
  const double* Cc = s->sum + (size_t)s->nblk * 36;
  const double* Kk = Cc + (size_t)F * 18;
  for (int i = 0; i < 6 * F; ++i)
    for (int k = 0; k < 3; ++k) { S[(size_t)i * NS + 6 * F + k] = Cc[3 * i + k]; S[(size_t)(6 * F + k) * NS + i] = Cc[3 * i + k]; }
  for (int a = 0; a < 3; ++a)
    for (int k = 0; k < 3; ++k) S[(size_t)(6 * F + a) * NS + 6 * F + k] = Kk[3 * a + k];
  for (int i = 0; i < NS; ++i)
    for (int j = 0; j < NS; ++j) S[(size_t)i * NS + j] = sblocks_fix(S[(size_t)i * NS + j], i, j, active, Dc);
}

/* band(+arrow) Cholesky solve of the merged blocks: x <- solution of (S + D^2) x = x.
   returns 0 ok, 1 not positive definite */
static int sblocks_band_solve(sblocks_t* s, int F, const unsigned char* active, const double* Dc, double* x) {
  const int nb = 6 * F, bw = 6 * s->span + 5 < nb - 1 ? 6 * s->span + 5 : nb - 1, LS = bw + 1;
  if (!s->AB) {
    s->AB = (double*)malloc(sizeof(double) * (size_t)nb * LS);
    s->AR = (double*)malloc(sizeof(double) * 3 * (size_t)nb);
    if (!s->AB || !s->AR) return 1;
  }
  double* AB = s->AB;
  double* AR = s->AR;
  memset(AB, 0, sizeof(double) * (size_t)nb * LS);
  for (int k = 0; k < s->nblk; ++k) {
    const int a = s->blk_a[k], b = s->blk_b[k];
    const double* B = s->sum + 36 * (size_t)k;
    for (int r = 0; r < 6; ++r)
      for (int c = 0; c < 6; ++c) {
        const int i = 6 * a + r, j = 6 * b + c;        /* upper element (i, j) when a < b */
        if (a == b && c > r) continue;                  /* diagonal block: lower part */
        const int hi = a == b ? i : j, lo = a == b ? j : i;
        AB[(size_t)hi * LS + (hi - lo)] = sblocks_fix(B[6 * r + c], hi, lo, active, Dc);
      }
  }
  /* an image without observations has no (a, a) block: its inactive slots still need their unit pivot */
  for (int i = 0; i < nb; ++i)
    if (!active[i]) AB[(size_t)i * LS] = 1.0;
  const double* Cc = s->sum + (size_t)s->nblk * 36;
  const double* Kk = Cc + (size_t)F * 18;
  for (int i = 0; i < nb; ++i)
    for (int k = 0; k < 3; ++k) AR[(size_t)k * nb + i] = sblocks_fix(Cc[3 * i + k], nb + k, i, active, Dc);
  double K3[9];
  for (int a = 0; a < 3; ++a)
    for (int k = 0; k < 3; ++k) K3[3 * a + k] = sblocks_fix(Kk[3 * a + k], nb + a, nb + k, active, Dc);
  /* L in place: row-oriented band Cholesky */
  for (int i = 0; i < nb; ++i) {
    const int j0 = i - bw > 0 ? i - bw : 0;
    double* Li = AB + (size_t)i * LS;
    for (int j = j0; j <= i; ++j) {
      const double* Lj = AB + (size_t)j * LS;
      const int k0 = (j - bw > j0) ? j - bw : j0;
      double v = Li[i - j];
      for (int k = k0; k < j; ++k) v -= Li[i - k] * Lj[j - k];
      if (i == j) {
        if (!(v > 0.0) || !isfinite(v)) return 1;
        Li[0] = sqrt(v);
      } else {
        Li[i - j] = v / Lj[0];
      }
    }
  }
  for (int a = 0; a < 3; ++a) {
    double* La = AR + (size_t)a * nb;
    for (int j = 0; j < nb; ++j) {
      const double* Lj = AB + (size_t)j * LS;
      const int k0 = j - bw > 0 ? j - bw : 0;
      double v = La[j];
      for (int k = k0; k < j; ++k) v -= La[k] * Lj[j - k];
      La[j] = v / Lj[0];
    }
  }
  for (int a = 0; a < 3; ++a)
    for (int k = 0; k <= a; ++k) {
      double v = K3[3 * a + k];
      for (int j = 0; j < nb; ++j) v -= AR[(size_t)a * nb + j] * AR[(size_t)k * nb + j];
      K3[3 * a + k] = v;
    }
  double Lk[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  for (int a = 0; a < 3; ++a)
    for (int k = 0; k <= a; ++k) {
      double v = K3[3 * a + k];
      for (int m = 0; m < k; ++m) v -= Lk[3 * a + m] * Lk[3 * k + m];
      if (a == k) {
        if (!(v > 0.0) || !isfinite(v)) return 1;
        Lk[3 * a + a] = sqrt(v);
      } else {
        Lk[3 * a + k] = v / Lk[3 * k + k];
      }
    }
  /* forward: L y = b */
  for (int i = 0; i < nb; ++i) {
    const double* Li = AB + (size_t)i * LS;
    const int j0 = i - bw > 0 ? i - bw : 0;
    double v = x[i];
    for (int j = j0; j < i; ++j) v -= Li[i - j] * x[j];
    x[i] = v / Li[0];
  }
  for (int a = 0; a < 3; ++a) {
    double v = x[nb + a];
    for (int j = 0; j < nb; ++j) v -= AR[(size_t)a * nb + j] * x[j];
    for (int m = 0; m < a; ++m) v -= Lk[3 * a + m] * x[nb + m];
    x[nb + a] = v / Lk[3 * a + a];
  }
  /* backward: L' x = y */
  for (int a = 2; a >= 0; --a) {
    double v = x[nb + a];
    for (int m = a + 1; m < 3; ++m) v -= Lk[3 * m + a] * x[nb + m];
    x[nb + a] = v / Lk[3 * a + a];
  }
  for (int i = nb - 1; i >= 0; --i) {
    double v = x[i];
    for (int a = 0; a < 3; ++a) v -= AR[(size_t)a * nb + i] * x[nb + a];
    const int j1 = i + bw < nb - 1 ? i + bw : nb - 1;
    for (int j = i + 1; j <= j1; ++j) v -= AB[(size_t)j * LS + (j - i)] * x[j];
    x[i] = v / AB[(size_t)i * LS];
  }
  return 0;
}

#endif
