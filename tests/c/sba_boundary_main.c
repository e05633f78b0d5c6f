/* tests/c/sba_boundary_main.c -- boundary test of the sba-1.5 drop-in (shim/sba_b200.c).
 * When the reference sources are at hand it is compiled against the REFERENCE's own lib/sba-1.5/sba.h (shim/Makefile,
 * BSFM_REFERENCE_SBA_H), so the calls below type-check against the reference declarations of sba_motstr_levmar /
 * sba_mot_levmar (sba.h:96-115); otherwise against the declarations below, which are those of shim/sba_b200.c.  Linked
 * against libsba_b200.so + libsfmdrv_b200.so instead of libsba.v1.5.a + libsfmdrv.a.
 *   sba_boundary_test <scene.bin> <result.bin> [mot]   solve the scene the way run_sfm does (sfm.c:652-838)
 *   sba_boundary_test foreign                          a foreign projection callback must fail loudly with SBA_ERROR
 * scene.bin : int32 n, m, nvis, est_focal, undistort | vmask n*m bytes | projections 2*nvis f64 | per camera R(9) t(3) f k(2) f64 | points 3n f64
 * result.bin: int32 rc | info 10 f64 | p (m*cnp + 3n) f64 */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#ifdef BSFM_REFERENCE_SBA_H
#include "sba.h"              /* the reference header */
#endif
#include "bsfm_b200_sba.h"    /* sfm_global_t mirror + the exported sfm_project_point3 */
#ifndef BSFM_REFERENCE_SBA_H
#define SBA_INFOSZ 10
#define SBA_ERROR (-1)
int sba_motstr_levmar(const int n, const int m, const int mcon, char *vmask, double *p, const int cnp, const int pnp,
                      double *x, double *covx, const int mnp,
                      void (*proj)(int j, int i, double *aj, double *bi, double *xij, void *adata),
                      void (*projac)(int j, int i, double *aj, double *bi, double *Aij, double *Bij, void *adata),
                      void *adata, const int itmax, const int verbose, const double *opts, double *info,
                      int use_constraints, bsfm_camera_constraints_t *constraints,
                      int use_point_constraints, bsfm_point_constraints_t *point_constraints,
                      double *Vout, double *Sout, double *Uout, double *Wout);
int sba_mot_levmar(const int n, const int m, const int mcon, char *vmask, double *p, const int cnp,
                   double *x, double *covx, const int mnp,
                   void (*proj)(int j, int i, double *aj, double *xij, void *adata),
                   void (*projac)(int j, int i, double *aj, double *Aij, void *adata),
                   void *adata, const int itmax, const int verbose, const double *opts, double *info,
                   int use_constraints, bsfm_camera_constraints_t *constraints);
#endif

static void foreign_proj(int j, int i, double *aj, double *bi, double *xij, void *adata)
{
    (void) j; (void) i; (void) aj; (void) adata;
    xij[0] = bi[0]; xij[1] = bi[1];
}

static void must_read(void *dst, size_t bytes, FILE *f)
{
    if (fread(dst, 1, bytes, f) != bytes) { fprintf(stderr, "short read\n"); exit(2); }
}

int main(int argc, char **argv)
{
    if (argc == 2 && !strcmp(argv[1], "foreign")) {
        char vmask[4] = {1, 1, 1, 1};
        double p[2 * 6 + 2 * 3] = {0}, x[8] = {0}, info[SBA_INFOSZ];
        double opts[6] = {1e-3, 1e-10, 1e-12, 1e-12, 0.0, 4e-2};
        int rc = sba_motstr_levmar(2, 2, 0, vmask, p, 6, 3, x, NULL, 2, foreign_proj, NULL, NULL, 10, 0, opts, info, 0, NULL, 0, NULL, NULL, NULL, NULL, NULL);
        printf("foreign rc=%d\n", rc);
        return rc == SBA_ERROR ? 0 : 1;
    }
    if (argc < 3) { fprintf(stderr, "usage: %s <scene.bin> <result.bin> [mot] | foreign\n", argv[0]); return 2; }
    const int mot = argc > 3 && !strcmp(argv[3], "mot");
    FILE *f = fopen(argv[1], "rb");
    if (!f) { perror(argv[1]); return 2; }
    int hdr[5];
    must_read(hdr, sizeof hdr, f);
    const int n = hdr[0], m = hdr[1], nvis = hdr[2], est_focal = hdr[3], undistort = hdr[4];
    char *vmask = malloc((size_t) n * m);
    double *x = malloc((size_t) nvis * 2 * sizeof(double));
    bsfm_camera_params_t *cams = calloc(m, sizeof *cams);
    bsfm_v3_t *pts = malloc((size_t) n * sizeof *pts);
    must_read(vmask, (size_t) n * m, f);
    must_read(x, (size_t) nvis * 2 * sizeof(double), f);
    for (int j = 0; j < m; j++) {
        double c[15];
        must_read(c, sizeof c, f);
        memcpy(cams[j].R, c, 9 * sizeof(double)); memcpy(cams[j].t, c + 9, 3 * sizeof(double));
        cams[j].f = c[12]; cams[j].k[0] = c[13]; cams[j].k[1] = c[14];
        cams[j].f_scale = 0.001; cams[j].k_scale = 5.0;       /* sfm.c:634-635, :656-657 */
    }
    must_read(pts, (size_t) n * sizeof *pts, f);
    fclose(f);
    const int cnp = 6 + (est_focal ? 1 : 0) + (undistort ? 2 : 0);
    const size_t np = (size_t) m * cnp + 3 * (size_t) n;
    double *p = calloc(np, sizeof(double));
    for (int j = 0; j < m; j++) {                            /* sfm.c:652-696 */
        int c = 6;
        memcpy(p + (size_t) cnp * j, cams[j].t, 3 * sizeof(double));
        if (est_focal) { p[(size_t) cnp * j + 6] = cams[j].f * cams[j].f_scale; c = 7; }
        if (undistort) { p[(size_t) cnp * j + c] = cams[j].k[0] * cams[j].k_scale; p[(size_t) cnp * j + c + 1] = cams[j].k[1] * cams[j].k_scale; }
    }
    memcpy(p + (size_t) m * cnp, pts, (size_t) n * 3 * sizeof(double));
    bsfm_sfm_global_t g;
    memset(&g, 0, sizeof g);
    g.num_cameras = m; g.num_points = n; g.num_params_per_camera = cnp;
    g.est_focal_length = est_focal; g.const_focal_length = 0; g.explicit_camera_centers = 1; g.estimate_distortion = undistort;
    g.init_params = cams; g.points = pts;
    double opts[6] = {1.0e-3, 1.0e-10, 1.0e-12, 1.0e-12, 0.0, 4.0e-2};     /* sfm.c:705-714 */
    double info[SBA_INFOSZ] = {0};
    int rc;
    if (mot)
        rc = sba_mot_levmar(n, m, 0, vmask, p, cnp, x, NULL, 2, sfm_project_point3_mot, NULL, &g, 150, 0, opts, info, 0, NULL);
    else
        rc = sba_motstr_levmar(n, m, 0, vmask, p, cnp, 3, x, NULL, 2, sfm_project_point3, NULL, &g, 150, 0, opts, info,
                               0, NULL, 0, NULL, NULL, NULL, NULL, NULL);
    /* the exported host projection agrees with the packed model: reproject observation 0 of point 0 */
    {
        int j0 = 0; while (j0 < m && !vmask[j0]) j0++;
        double xij[2];
        if (j0 < m) { sfm_project_point3(j0, 0, p + (size_t) cnp * j0, p + (size_t) m * cnp, xij, &g); printf("reproj0 %.6f %.6f (measured %.6f %.6f)\n", xij[0], xij[1], x[0], x[1]); }
    }
    FILE *o = fopen(argv[2], "wb");
    if (!o) { perror(argv[2]); return 2; }
    fwrite(&rc, sizeof rc, 1, o); fwrite(info, sizeof(double), SBA_INFOSZ, o); fwrite(p, sizeof(double), np, o);
    fclose(o);
    printf("rc=%d iterations=%d stop=%d\n", rc, (int) info[5], (int) info[6]);
    return rc >= 0 ? 0 : 1;
}
