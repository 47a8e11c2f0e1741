// Host build of igd_g711_transcode1 (igate4xsoftphonedsp_b200/csrc/igd_math.cuh, -DIGD_HOST_EMUL): the code table
// k_fanout_pkt_tile builds per CTA.  TEST-ONLY: it is never loaded by the product.
#define IGD_HOST_EMUL 1
#include "../../include/igate_dsp.h"
#include "../../igate4xsoftphonedsp_b200/csrc/igd_math.cuh"

extern "C" void emul_transcode_table(unsigned char *out /* [in law][out law][256] */)
{
    for (int k = 0; k < 4; k++)
        for (unsigned c = 0; c < 256; c++) out[k * 256 + c] = (unsigned char)igd_g711_transcode1(c, k >> 1, k & 1);
}
