/*
 * gps.h -- the declarations of the receiver's gps/gps.h that the adapter (integration/search_gpu.cpp) and the test
 * receiver (integration/harness_gpu.cpp) use, restated so that the adapter builds and runs its tests from this
 * repository alone.  integration/Makefile compiles against this directory by default; `make REF=<FlyDog_SDR_GPS tree>`
 * compiles against the receiver's own gps/gps.h, types.h and gps/sats.cpp instead, where a drift of any prototype
 * below is a build error.
 *
 * Names, prototypes, default arguments and the leading SATELLITE members follow gps/gps.h; the constants are the
 * receiver's (FS = 16.368 MHz, one 65536-sample capture block, decimation by 4, 249.76 Hz Doppler bins).
 */
#pragma once
#include "types.h"
#include "kiwi.h"

#define FS 16.368e6
#define NSAMPLES 65536                 /* 1-bit samples per capture block (4.004 ms) */
#define DECIM 4
#define BIN_SIZE (FS / NSAMPLES)       /* 249.755859375 Hz */
#define MAX_SATS 64

enum sat_e { Navstar = 0, SBAS = 1, QZSS = 2, E1B = 3 };

struct SATELLITE {
    int prn, T1, T2;                   /* QZSS rows: T1 = G2 delay, T2 = G2 initial state */
    sat_e type;
    int sat;                           /* row index, set by SearchInit */
    bool busy;
    char *prn_s;                       /* label set by SearchInit: "N01 ", "Q194", "E02 " */
};

extern SATELLITE Sats[];               /* gps/sats.cpp; ends with a row whose prn is -1 */

struct gps_t {
    int n_Navstar, n_QZSS, n_E1B;
    int acq_Navstar, acq_QZSS, acq_Galileo;
    int good;
};
extern gps_t gps;

enum STAT { STAT_PARAMS, STAT_SAT, STAT_DOP, STAT_ACQUIRE };

void SearchInit();
void SearchFree();
void SearchTask(void *param);
void SearchTaskRun();
void SearchEnable(int sat);
void SearchParams(int argc, char *argv[]);

int ChanReset(int sat, int codegen_init);
void ChanStart(int ch, int sat, int t_sample, int lo_shift, int ca_shift, int snr);

void GPSstat_init();
void GPSstat(STAT st, double d, int i = 0, int j = 0, int k = 0, int m = 0, double d2 = 0);
