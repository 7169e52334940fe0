// sats.cpp -- the receiver's satellite table (gps/sats.cpp) for the adapter's tests: the 59 rows of
// flydog_sdr_gps_b200/sats.py reference_table(), in the same order (sat = row index).
//   Navstar PRN 1..32: the G2 phase-select tap pair (IS-GPS-200 Table 3-Ia)
//   QZSS 194, 195, 196, 199: G2 delay and G2 initial state (IS-QZSS)
//   Galileo E1-B: the PRN of the memory code; the 23 satellites in active service
#include "types.h"
#include "gps.h"

SATELLITE Sats[] = {
    {1, 2, 6, Navstar},   {2, 3, 7, Navstar},   {3, 4, 8, Navstar},   {4, 5, 9, Navstar},
    {5, 1, 9, Navstar},   {6, 2, 10, Navstar},  {7, 1, 8, Navstar},   {8, 2, 9, Navstar},
    {9, 3, 10, Navstar},  {10, 2, 3, Navstar},  {11, 3, 4, Navstar},  {12, 5, 6, Navstar},
    {13, 6, 7, Navstar},  {14, 7, 8, Navstar},  {15, 8, 9, Navstar},  {16, 9, 10, Navstar},
    {17, 1, 4, Navstar},  {18, 2, 5, Navstar},  {19, 3, 6, Navstar},  {20, 4, 7, Navstar},
    {21, 5, 8, Navstar},  {22, 6, 9, Navstar},  {23, 1, 3, Navstar},  {24, 4, 6, Navstar},
    {25, 5, 7, Navstar},  {26, 6, 8, Navstar},  {27, 7, 9, Navstar},  {28, 8, 10, Navstar},
    {29, 1, 6, Navstar},  {30, 2, 7, Navstar},  {31, 3, 8, Navstar},  {32, 4, 9, Navstar},

    {194, 208, 01607, QZSS}, {195, 711, 01747, QZSS}, {196, 189, 01305, QZSS}, {199, 663, 0727, QZSS},

    {2, 0, 0, E1B},  {3, 0, 0, E1B},  {4, 0, 0, E1B},  {5, 0, 0, E1B},  {7, 0, 0, E1B},  {8, 0, 0, E1B},
    {9, 0, 0, E1B},  {10, 0, 0, E1B}, {11, 0, 0, E1B}, {12, 0, 0, E1B}, {13, 0, 0, E1B}, {15, 0, 0, E1B},
    {19, 0, 0, E1B}, {21, 0, 0, E1B}, {24, 0, 0, E1B}, {25, 0, 0, E1B}, {26, 0, 0, E1B}, {27, 0, 0, E1B},
    {30, 0, 0, E1B}, {31, 0, 0, E1B}, {33, 0, 0, E1B}, {34, 0, 0, E1B}, {36, 0, 0, E1B},

    {-1}
};
