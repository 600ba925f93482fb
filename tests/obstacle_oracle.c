/*
 * obstacle_oracle.c -- CPU oracle of the step with solid obstacles (TEST INFRASTRUCTURE ONLY).
 *
 * Obstacles have no counterpart in the reference, so this is not part of oracle/smoke_oracle.c, whose functions stay pinned to
 * the reference's golden vectors.  It includes that file and adds the obstacle variants on top of its phases, in the same
 * style: one statement per rounded fp32 operation, built with -ffp-contract=off (tests/obstacle_oracle.py builds and loads it).
 *
 * Semantics (DESIGN.md s5.7): a mask S marks solid cells.  One step is smk_oracle_step with
 *   O1  closed faces of u and v := +0.0 after the diffusions, then the divergence as usual;
 *   the Jacobi sweeps with Neumann ghost values at solid neighbours, solid cells and the ring := +0.0;
 *   the gradient subtract on open faces only;
 *   O4  closed faces of the advected u and v := +0.0, before the density advection;
 *   O3  the density (and so the frame) of solid cells := +0.0 after the decay.
 */
#include "../oracle/smoke_oracle.c"

/* ---- extension (no reference counterpart): solid obstacles ------------------------------------------
 * S[h][w] (uint8, 0 fluid / 1 solid, dense).  u face (i, j), 0 <= i <= h, lies between cells (i-1, j) and (i, j); v face (i, j),
 * 0 <= j <= w, between (i, j-1) and (i, j).  A face is closed when a cell it touches (that exists) is solid. */
static inline int u_closed(const unsigned char* S, int h, int w, int i, int j)
{
    return (i >= 1 && S[(long)(i - 1) * w + j]) || (i < h && S[(long)i * w + j]);
}
static inline int v_closed(const unsigned char* S, int h, int w, int i, int j)
{
    (void)h;
    return (j >= 1 && S[(long)i * w + j - 1]) || (j < w && S[(long)i * w + j]);
}
/* closed faces of u and v := +0.0 (a store: -x*0 would be -0, inf*0 NaN) */
static void close_faces(float* U, float* V, const unsigned char* S, int h, int w)
{
    for (int i = 0; i <= h; ++i) for (int j = 0; j < w; ++j) if (u_closed(S, h, w, i, j)) U[(long)i * w + j] = 0.0f;
    for (int i = 0; i < h; ++i) for (int j = 0; j <= w; ++j) if (v_closed(S, h, w, i, j)) V[(long)i * (w + 1) + j] = 0.0f;
}

/* K Jacobi sweeps with solid cells: a fluid interior cell takes a solid neighbour's value as its own p (Neumann ghost); solid
 * cells and the ring get +0.0.  With no solid cell this is smk_oracle_jacobi bit for bit. */
API void smk_oracle_jacobi_obst(float* P, const float* div, const unsigned char* S, float* tmp, int h, int w, int K)
{
    float* a = P; float* b = tmp;
    for (int k = 0; k < K; ++k) {
        memset(b, 0, sizeof(float) * (size_t)h * w);
        for (int i = 1; i < h - 1; ++i) for (int j = 1; j < w - 1; ++j) {
            const long c = (long)i * w + j;
            if (S[c]) continue;
            const float pc = a[c];
            const float qn = S[c - w] ? pc : a[c - w];
            const float qs = S[c + w] ? pc : a[c + w];
            const float qw = S[c - 1] ? pc : a[c - 1];
            const float qe = S[c + 1] ? pc : a[c + 1];
            float s = qn + qs;
            s = s + qw;
            s = s + qe;
            s = s - div[c];
            b[c] = 0.25f * s;
        }
        float* t = a; a = b; b = t;
    }
    if (a != P) memcpy(P, a, sizeof(float) * (size_t)h * w);
}

/* smk_oracle_step with solid cells S: O1 (close faces) after the diffusions, the masked Jacobi, the gradient subtract on open
 * faces only, O4 (close the advected u, v) before the density advection, O3 (solid density and frame := +0) at the end.
 * norms: {max, l2} of the post-projection divergence over interior fluid cells. */
API void smk_oracle_step_obst(float* U, float* V, float* P, float* D, int h, int w,
                              float dt, float c_uv, float c_d, int K,
                              float* work, float* frame, double* norms, const unsigned char* S)
{
    const long nu = (long)(h + 1) * w, nv = (long)h * (w + 1), nc = (long)h * w;
    float* t0 = work; float* t1 = work + (long)(h + 1) * (w + 1);
    smk_oracle_buoyancy(V, D, h, w, dt);
    smk_oracle_diffuse(U, t0, h + 1, w, c_uv); memcpy(U, t0, sizeof(float) * nu);
    smk_oracle_diffuse(V, t0, h, w + 1, c_uv); memcpy(V, t0, sizeof(float) * nv);
    smk_oracle_diffuse(D, t0, h, w, c_d);      memcpy(D, t0, sizeof(float) * nc);
    close_faces(U, V, S, h, w);                                                    /* O1 */
    smk_oracle_divergence(U, V, t0, h, w, dt);
    smk_oracle_jacobi_obst(P, t0, S, t1, h, w, K);
    for (int i = 1; i < h; ++i) for (int j = 0; j < w; ++j) {                      /* gradient subtract, open faces */
        if (u_closed(S, h, w, i, j)) continue;
        float g = P[(long)i * w + j] - P[(long)(i - 1) * w + j];
        float t = dt * g;
        U[(long)i * w + j] = U[(long)i * w + j] - t;
    }
    for (int i = 0; i < h; ++i) for (int j = 1; j < w; ++j) {
        if (v_closed(S, h, w, i, j)) continue;
        float g = P[(long)i * w + j] - P[(long)i * w + j - 1];
        float t = dt * g;
        V[(long)i * (w + 1) + j] = V[(long)i * (w + 1) + j] - t;
    }
    if (norms) {
        double mx = 0.0, ss = 0.0;
        for (int i = 1; i < h - 1; ++i) for (int j = 1; j < w - 1; ++j) {
            if (S[(long)i * w + j]) continue;
            float s = U[(long)(i + 1) * w + j] - U[(long)i * w + j];
            s = s + V[(long)i * (w + 1) + j + 1];
            s = s - V[(long)i * (w + 1) + j];
            double a = fabs((double)s); if (a > mx) mx = a; ss += (double)s * (double)s;
        }
        norms[0] = mx; norms[1] = sqrt(ss);
    }
    smk_oracle_advect(U, t0, h + 1, w, U, V, h, w, dt); memcpy(U, t0, sizeof(float) * nu);
    smk_oracle_advect(V, t0, h, w + 1, U, V, h, w, dt); memcpy(V, t0, sizeof(float) * nv);
    close_faces(U, V, S, h, w);                                                    /* O4 */
    smk_oracle_advect(D, t0, h, w, U, V, h, w, dt);
    for (long k = 0; k < nc; ++k) D[k] = t0[k] * 0.995f;
    for (long k = 0; k < nc; ++k) if (S[k]) D[k] = 0.0f;                           /* O3 */
    if (frame) memcpy(frame, D, sizeof(float) * nc);
}

