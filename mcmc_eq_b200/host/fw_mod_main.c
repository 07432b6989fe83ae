/* fw_mod_main.c -- the reference's forward programs `fw_mod` and `fw` on top of the B200 library (plain C over the C ABI).
 *
 *     fw_mod <config_eqx.dat> <model_block> <picks> [-d device] [-x]
 *     fw     <config.dat>     <res.dat>     <picks> [-d device] [-x]   (this file compiled with -DFW_GRIDDED)
 *
 * Arguments as the reference's.  fw_mod (src/fw_mod.c): <model_block> is one record cut from a chain file: the "mod ..."
 * line (src/fw_mod.c:421-445), then one "EQ ..." line per event (:450-457) and one "RES ..." line per station (:460-464).
 * fw (src/fw.c:405-455): <res.dat> is an analyse_eq result file: nz "STAN" lines (depth, ..., Vp = 7th and Vp/Vs = 9th
 * token) that become nz nuclei, one "EQ" line per event, as many "EZ" lines (skipped), one "RES" line per station in
 * station order, one noise line -- what Example/make_synthetics and scriptsV2/mkSynthetics.sh build to make synthetic picks.
 * Output as cal_fit_newx prints it with out == 1 (src/misfit.c:130-143): per event
 *     EVENT i  reftime x y z origin
 * and per pick (P first, then S, file order)
 *     residual dist z origin t_observed t_predicted P|S
 * and on stderr "Start model found with loglikelihood ... RMS=..." (src/fw_mod.c:480).  make_synthetics / mkSynthetics.sh /
 * disp_msft_dist.sh use exactly these lines.
 * -x: the same forward with reciprocal travel-time tables (mq_set_tables, MQ_TABLES_RECIPROCAL; one stderr line says so).
 * Comparing the output with and without -x on one's own picks shows what the mode costs per pick on that data.
 */
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/mcmceq_b200.h"
#include "mq_io.h"

#define FAIL(...) do { fprintf(stderr, __VA_ARGS__); fprintf(stderr, "\n"); rc = 1; goto done; } while (0)
#define MQ(call) do { int rc_ = (call); if (rc_ != MQ_OK) FAIL("%s failed (%d): %s", #call, rc_, mq_last_error()); } while (0)

/* src/mcmc_eq.c:1303-1306 */
static float dst(float x1, float x2, float y1, float y2) { return (float)sqrt(((x1 - x2) * (x1 - x2)) + ((y1 - y2) * (y1 - y2))); }

int main(int argc, char** argv)
{
    int rc = 0, device = 0, i, j, dim = 0, ne, ns, np, reciprocal = 0;
    mq_config cfg;
    mqio_picks pk;
    mq_handle* h = NULL;
    mq_models m;
    FILE* f = NULL;
    char* buf = NULL;
    const size_t cap = 5000 * 3 * 20;
    int32_t dim32;
    float *z = NULL, *vp = NULL, *vpvs = NULL, *eq = NULL, *pres = NULL, *sres = NULL, *origin = NULL, *resid = NULL, *tpred = NULL;
    float noise[8], mf[8];
    double misfit, rms;

    memset(&pk, 0, sizeof pk);
    memset(&m, 0, sizeof m);
    if (argc < 4) { fprintf(stderr, "usage: %s config.dat model picks [-d device] [-x]\n", argv[0]); return 2; }
    for (i = 4; i < argc; i++) {
        if (!strcmp(argv[i], "-d") && i + 1 < argc) device = atoi(argv[++i]);
        else if (!strcmp(argv[i], "-x")) reciprocal = 1;
    }
    if (mqio_read_config(argv[1], &cfg) != MQ_OK) FAIL("%s", mqio_last_error());
    if (mqio_read_picks(argv[3], &pk) != MQ_OK) FAIL("%s", mqio_last_error());
    ne = pk.view.n_events; ns = pk.view.n_stations; np = pk.view.n_picks;

    if (!(f = fopen(argv[2], "r"))) FAIL("could not open model file %s", argv[2]);
    buf = (char*)malloc(cap);
    z = (float*)calloc(1000, sizeof(float)); vp = (float*)calloc(1000, sizeof(float)); vpvs = (float*)calloc(1000, sizeof(float));
    eq = (float*)calloc((size_t)ne * 3, sizeof(float)); origin = (float*)calloc((size_t)ne, sizeof(float));
    pres = (float*)calloc((size_t)ns, sizeof(float)); sres = (float*)calloc((size_t)ns, sizeof(float));
    resid = (float*)calloc((size_t)np, sizeof(float)); tpred = (float*)calloc((size_t)np, sizeof(float));
    if (!buf || !z || !vp || !vpvs || !eq || !origin || !pres || !sres || !resid || !tpred) FAIL("out of memory");
    if (!fgets(buf, (int)cap, f)) FAIL("empty model file %s", argv[2]);
#ifdef FW_GRIDDED
    {   /* src/fw.c:405-455 */
        int k;
        char a[64];
        float t[11];
        dim = cfg.grid.nz;
        if (dim > 1000) FAIL("nz %d > 1000 nuclei", dim);
        for (k = 0; k < 8; k++) noise[k] = cfg.start_noise > 0.f ? cfg.start_noise : 1.f;
        for (k = 0; k < dim; k++) {
            if (k > 0 && !fgets(buf, (int)cap, f)) FAIL("model file: STAN line %d missing", k);
            if (sscanf(buf, "%63s %f %f %f %f %f %f %f %f", a, &t[0], &t[1], &t[2], &t[3], &t[4], &t[5], &t[6], &t[7]) < 9)
                FAIL("model file: STAN line %d short", k);
            z[k] = t[0]; vp[k] = t[5]; vpvs[k] = t[7];
        }
        for (i = 0; i < ne; i++) {   /* "EQ i x y z . . . . origin ." */
            int di;
            if (!fgets(buf, (int)cap, f) || sscanf(buf, "%63s %d %f %f %f %f %f %f %f %f", a, &di, &eq[3 * i], &eq[3 * i + 1], &eq[3 * i + 2],
                                                    &t[0], &t[1], &t[2], &t[3], &origin[i]) < 5)
                FAIL("model file: EQ line %d missing or short", i);
        }
        for (i = 0; i < ne; i++)
            if (!fgets(buf, (int)cap, f)) FAIL("model file: EZ line %d missing", i);
        for (i = 0; i < ns; i++) {   /* "RES i pres sres . ." -- by line order, like the reference */
            int di;
            if (!fgets(buf, (int)cap, f) || sscanf(buf, "%63s %d %f %f", a, &di, &pres[i], &sres[i]) < 4)
                FAIL("model file: RES line %d missing or short", i);
        }
    }
#else
    {   /* "mod XX number dim rms p0 p1 p2 p3 s0 s1 s2 s3 z vp vpvs ..." (src/fw_mod.c:421-445) */
        char* tok = strtok(buf, " ");
        float pn[8];
        int k;
        tok = strtok(NULL, " ");                                  /* type */
        tok = strtok(NULL, " ");                                  /* model number */
        tok = strtok(NULL, " "); if (!tok) FAIL("bad model line"); dim = atoi(tok);
        tok = strtok(NULL, " ");                                  /* rms */
        for (k = 0; k < 8; k++) { tok = strtok(NULL, " "); if (!tok) FAIL("bad model line"); pn[k] = (float)atof(tok); }
        for (k = 0; k < 4; k++) { noise[2 * k] = pn[k]; noise[2 * k + 1] = pn[4 + k]; }   /* file: p0..p3 s0..s3 */
        if (dim < 1 || dim > 1000) FAIL("bad model dimension %d", dim);
        for (k = 0; k < dim; k++) {
            char *a = strtok(NULL, " "), *b = strtok(NULL, " "), *c = strtok(NULL, " ");
            if (!a || !b || !c) FAIL("model line ends after %d of %d nuclei", k, dim);
            z[k] = (float)atof(a); vp[k] = (float)atof(b); vpvs[k] = (float)atof(c);
        }
    }
    for (i = 0; i < ne; i++) {   /* "EQ XX number i rms x y z reftime origin" */
        char a[64], b[64];
        int d1, d2;
        float df, dg;
        if (!fgets(buf, (int)cap, f) || sscanf(buf, "%63s %63s %d %d %f %f %f %f %f %f", a, b, &d1, &d2, &df, &eq[3 * i], &eq[3 * i + 1],
                                                &eq[3 * i + 2], &origin[i], &dg) < 8)
            FAIL("model file: EQ line %d missing or short", i);
    }
    for (i = 0; i < ns; i++) {   /* "RES XX number i rms pres sres" */
        char a[64], b[64];
        int d1, d2;
        float df;
        if (!fgets(buf, (int)cap, f) || sscanf(buf, "%63s %63s %d %d %f %f %f", a, b, &d1, &d2, &df, &pres[i], &sres[i]) < 7)
            FAIL("model file: RES line %d missing or short", i);
    }

#endif
    if (cfg.max_dim < dim) cfg.max_dim = dim;      /* the reference's forward programs do not look at line 8 */
    MQ(mq_create(&cfg, &pk.view, 1, device, 1, &h));
    if (reciprocal) {
        MQ(mq_set_tables(h, MQ_TABLES_RECIPROCAL));
        fprintf(stderr, "reciprocal travel-time tables (-x): sources at the receiver rows, not the parity forward\n");
    }
    dim32 = dim;
    m.n_chains = 1; m.max_dim = dim; m.n_events = ne; m.n_stations = ns;
    m.dim = &dim32; m.z = z; m.vp = vp; m.vpvs = vpvs; m.eq = eq; m.pres = pres; m.sres = sres; m.noise = noise; m.origin = origin;
    fprintf(stderr, "Start misfit calc\n");
    MQ(mq_forward_host(h, &m, 3, mf, origin));
    MQ(mq_get_predictions(h, 0, resid, tpred));
    for (i = 0; i < ne; i++) {
        const int b = pk.ev_off[i], e = pk.ev_off[i + 1];
        printf("EVENT %d  %lf %f %f %f %f\n", i, pk.reftime[i], eq[3 * i], eq[3 * i + 1], eq[3 * i + 2], origin[i]);
        for (j = b; j < e; j++)
            printf("%f %f %f %f %f %f %c\n", resid[j], dst(pk.x[j], eq[3 * i], pk.y[j], eq[3 * i + 1]), eq[3 * i + 2], origin[i], pk.t[j],
                   tpred[j], (j - b) < pk.n_p[i] ? 'P' : 'S');
    }
    /* src/fw_mod.c:470-480.  cal_fit_newx always returns 1.0 (src/misfit.c:160) and fw_mod takes that return value for
     * the misfit, so the reference prints "loglikelihood -0.500000" whatever the model; scripts only read the RMS. */
    misfit = 1.0;
    rms = sqrt((double)((((((((mf[0] + mf[2]) + mf[4]) + mf[6]) + mf[1]) + mf[3]) + mf[5]) + mf[7]) / (float)np));
    fprintf(stderr, "Start model found with loglikelihood %f RMS=%f\n", -misfit / 2.0, rms);

done:
    if (f) fclose(f);
    if (h) mq_destroy(h);
    free(buf); free(z); free(vp); free(vpvs); free(eq); free(origin); free(pres); free(sres); free(resid); free(tpred);
    mqio_free_picks(&pk);
    return rc;
}
