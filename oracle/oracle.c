/*
 * oracle/oracle.c -- TEST INFRASTRUCTURE (CPU restatement), never shipped, never imported by the product.
 *
 * Plain-C restatement of the arithmetic of VVenC's block-cost hot path, written from the definitions
 * (SURVEY.md section 8a), each function citing the reference file:line it follows.  It is pinned against the
 * reference's own scalar and AVX2 kernels (oracle/_ref, built by oracle/Makefile.ref) by
 * tests/test_oracle_vs_reference.py, and against the committed vectors in tests/golden/ everywhere else.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load this.
 */
#include <stdint.h>
#include <stddef.h>
#include <stdlib.h>
#include <string.h>
#include <math.h>
#include "vvc_tables.h"
#include "vvc_lfnst_tables.h"

typedef int16_t Pel;

static inline int iabs( int v ) { return v < 0 ? -v : v; }
static inline int ilog2u( uint32_t v ) { int r = 0; while( v > 1 ) { v >>= 1; r++; } return r; }

int orc_version( void ) { return 1; }

/* ------------------------------------------------------------------------------------------------------
 * SAD  (CommonLib/RdCost.cpp:300-335 xGetSAD; width-specialised :337-644 compute the same sum)
 * rows visited with step 2^subShift, result << subShift.  Early exit is not modelled: callers of the
 * reference use maximumDistortionForEarlyExit = MAX_DISTORTION for comparison (vvenc_unit_test.cpp:1957).
 * ---------------------------------------------------------------------------------------------------- */
uint64_t orc_sad( const Pel* org, int so, const Pel* cur, int sc, int w, int h, int subShift )
{
  const int step = 1 << subShift;
  uint64_t sum = 0;
  for( int y = 0; y < h; y += step )
    for( int x = 0; x < w; x++ )
      sum += (uint64_t) iabs( org[y * so + x] - cur[y * sc + x] );
  return sum << subShift;
}

/* SSE (CommonLib/RdCost.cpp:651-1000): sum of squared differences, no sub-sampling, 64-bit */
uint64_t orc_sse( const Pel* org, int so, const Pel* cur, int sc, int w, int h )
{
  uint64_t sum = 0;
  for( int y = 0; y < h; y++ )
    for( int x = 0; x < w; x++ )
    {
      const int d = org[y * so + x] - cur[y * sc + x];
      sum += (uint64_t)( d * d );
    }
  return sum;
}

/* ------------------------------------------------------------------------------------------------------
 * SATD.  A tile's cost is sum|H_th * D * H_tw| with the DC term down-weighted, then a shape-dependent
 * normalisation (CommonLib/RdCost.cpp: 2x2 :1006-1026, 4x4 :1028-1124, 8x8 :1225-1322, 16x8 :1324-1470,
 * 8x16 :1472-1609, 4x8 :1611-1685, 8x4 :1687-1766, 16x16_fast :1126-1223).  The reference's butterfly order
 * only permutes/negates Hadamard outputs, so sum|.| and |DC| are order independent.
 * ---------------------------------------------------------------------------------------------------- */
static void wht1d( int* v, int n, int stride )
{
  for( int len = 1; len < n; len <<= 1 )
    for( int i = 0; i < n; i += len << 1 )
      for( int j = i; j < i + len; j++ )
      {
        const int a = v[j * stride], b = v[( j + len ) * stride];
        v[j * stride] = a + b; v[( j + len ) * stride] = a - b;
      }
}

static uint64_t had_tile( const int* diff, int tw, int th )
{
  int m[16 * 16];
  memcpy( m, diff, sizeof( int ) * tw * th );
  for( int y = 0; y < th; y++ ) wht1d( m + y * tw, tw, 1 );
  for( int x = 0; x < tw; x++ ) wht1d( m + x, th, tw );
  int64_t sad = 0;
  for( int i = 0; i < tw * th; i++ ) sad += iabs( m[i] );
  const int dc = iabs( m[0] );
  if( tw == 2 && th == 2 )                      /* :1020-1023: only the DC term is scaled, no final normalisation */
    return (uint64_t)( sad - dc + ( dc >> 2 ) );
  sad = sad - dc + ( dc >> 2 );
  if( tw == 4 && th == 4 ) return (uint64_t)( ( sad + 1 ) >> 1 );                    /* :1121 */
  if( tw == 8 && th == 8 ) return (uint64_t)( ( sad + 2 ) >> 2 );                    /* :1319 */
  if( tw * th == 128 )     return (uint64_t)(int)( (int) sad / sqrt( 16.0 * 8 ) * 2 );  /* :1467,1606 */
  if( tw * th == 32 )      return (uint64_t)(int)( (int) sad / sqrt( 4.0 * 8 ) * 2 );   /* :1682,1763 */
  return 0;
}

static uint64_t had_tile_at( const Pel* org, int so, const Pel* cur, int sc, int tw, int th )
{
  int diff[16 * 16];
  for( int y = 0; y < th; y++ )
    for( int x = 0; x < tw; x++ )
      diff[y * tw + x] = org[y * so + x] - cur[y * sc + x];
  return had_tile( diff, tw, th );
}

/* 16x16 'fast': 2x2 rounded means of org and cur separately, 8x8 Hadamard, ((sad+2)>>2)<<2 (:1126-1223) */
static uint64_t had_tile16_fast( const Pel* org, int so, const Pel* cur, int sc )
{
  int diff[64];
  for( int y = 0; y < 8; y++ )
    for( int x = 0; x < 8; x++ )
    {
      const Pel* o = org + 2 * y * so + 2 * x;
      const Pel* c = cur + 2 * y * sc + 2 * x;
      diff[y * 8 + x] = ( ( o[0] + o[1] + o[so] + o[so + 1] + 2 ) >> 2 ) - ( ( c[0] + c[1] + c[sc] + c[sc + 1] + 2 ) >> 2 );
    }
  return had_tile( diff, 8, 8 ) << 2;
}

/* tile choice: CommonLib/RdCost.cpp:1818-1938 (xGetHADs<fastHad>) */
uint64_t orc_had( const Pel* org, int so, const Pel* cur, int sc, int w, int h, int fast )
{
  int tw, th, f16 = 0;
  if(      w > h && ( h & 7 ) == 0 && ( w & 15 ) == 0 ) { tw = 16; th = 8; }
  else if( w < h && ( w & 7 ) == 0 && ( h & 15 ) == 0 ) { tw = 8;  th = 16; }
  else if( w > h && ( h & 3 ) == 0 && ( w & 7 ) == 0 )  { tw = 8;  th = 4; }
  else if( w < h && ( w & 3 ) == 0 && ( h & 7 ) == 0 )  { tw = 4;  th = 8; }
  else if( fast && ( h % 32 == 0 ) && ( w % 32 == 0 ) && w == h ) { tw = 16; th = 16; f16 = 1; }
  else if( ( h % 8 == 0 ) && ( w % 8 == 0 ) ) { tw = 8; th = 8; }
  else if( ( h % 4 == 0 ) && ( w % 4 == 0 ) ) { tw = 4; th = 4; }
  else if( ( h % 2 == 0 ) && ( w % 2 == 0 ) ) { tw = 2; th = 2; }
  else return UINT64_MAX;                       /* reference THROWs "Invalid size" */
  uint64_t sum = 0;
  for( int y = 0; y < h; y += th )
    for( int x = 0; x < w; x += tw )
      sum += f16 ? had_tile16_fast( org + y * so + x, so, cur + y * sc + x, sc )
                 : had_tile_at( org + y * so + x, so, cur + y * sc + x, sc, tw, th );
  return sum;
}

/* min(SATD, 2*SAD) (CommonLib/RdCost.cpp:1768-1816); the reference requires compact buffers, the value is
 * defined for any stride */
uint64_t orc_had2sad( const Pel* org, int so, const Pel* cur, int sc, int w, int h )
{
  const uint64_t had = orc_had( org, so, cur, sc, w, h, 0 );
  const uint64_t sad = orc_sad( org, so, cur, sc, w, h, 0 );
  return had < 2 * sad ? had : 2 * sad;
}

/* family: 0 SSE, 1 SAD, 2 HAD, 3 HAD_fast, 4 HAD_2SAD */
uint64_t orc_dist( int family, const Pel* org, int so, const Pel* cur, int sc, int w, int h, int subShift )
{
  switch( family )
  {
    case 0: return orc_sse( org, so, cur, sc, w, h );
    case 1: return orc_sad( org, so, cur, sc, w, h, subShift );
    case 2: return orc_had( org, so, cur, sc, w, h, 0 );
    case 3: return orc_had( org, so, cur, sc, w, h, 1 );
    case 4: return orc_had2sad( org, so, cur, sc, w, h );
  }
  return UINT64_MAX;
}

void orc_dist_list( int family, const Pel* orgPlane, int so, const Pel* curPlane, int sc, const int32_t* desc, int n, int subShift, uint64_t* out )
{
  for( int i = 0; i < n; i++ )
  {
    const int32_t* d = desc + 6 * (size_t) i;
    out[i] = orc_dist( family, orgPlane + (ptrdiff_t) d[1] * so + d[0], so, curPlane + (ptrdiff_t) d[3] * sc + d[2], sc, d[4], d[5], subShift );
  }
}

/* GEO mask-weighted SAD (CommonLib/RdCost.cpp:2062-2093) */
uint64_t orc_sad_mask( const Pel* org, int so, const Pel* cur, int sc, int w, int h, const Pel* mask, int maskStride, int stepX, int maskStride2, int subShift )
{
  const int step = 1 << subShift;
  uint64_t sum = 0;
  for( int y = 0; y < h; y += step )
  {
    for( int x = 0; x < w; x++ ) { sum += (uint64_t)( iabs( org[x] - cur[x] ) * *mask ); mask += stepX; }
    org += so * step; cur += sc * step; mask += maskStride * step; mask += maskStride2;
  }
  return sum << subShift;
}

/* DMVR row of five SADs (CommonLib/RdCost.cpp:1984-2034): position i uses org+i and cur-i, each >>1 */
void orc_sad_x5( const Pel* org, int so, const Pel* cur, int sc, int w, int h, int subShift, int calcCentre, uint64_t* cost5 )
{
  for( int i = 0; i < 5; i++ )
  {
    if( i == 2 && !calcCentre ) continue;
    cost5[i] = orc_sad( org + i, so, cur - i, sc, w, h, subShift ) >> 1;
  }
}

/* fixed-weight SSE (CommonLib/RdCost.cpp:1942-1982): sum((w*d*d + 2^15) >> 16), odd width only for w==1 */
uint64_t orc_fix_wsse( const Pel* org, int so, const Pel* cur, int sc, int w, int h, uint32_t weight )
{
  uint64_t sum = 0;
  for( int y = 0; y < h; y++ )
    for( int x = 0; x < w; x++ )
    {
      const int32_t d = org[y * so + x] - cur[y * sc + x];
      sum += (uint64_t)(int32_t)( ( (int64_t) weight * ( d * d ) + ( 1 << 15 ) ) >> 16 );
    }
  return sum;
}

/* ------------------------------------------------------------------------------------------------------
 * MV rate (CommonLib/RdCost.h:181-203)
 * ---------------------------------------------------------------------------------------------------- */
static uint32_t eg_bits( int v )
{
  const uint32_t t = v <= 0 ? ( (uint32_t)( -v ) << 1 ) + 1 : (uint32_t) v << 1;
  return 1 + ( (uint32_t) ilog2u( t ) << 1 );
}

uint32_t orc_mv_bits( int x, int y, int predHor, int predVer, int costScale, int imvShift )
{
  return eg_bits( ( x * ( 1 << costScale ) - predHor ) >> imvShift ) + eg_bits( ( y * ( 1 << costScale ) - predVer ) >> imvShift );
}

uint64_t orc_mv_cost( double lambda, int x, int y, int predHor, int predVer, int costScale, int imvShift )
{
  const double motionLambda = sqrt( lambda );       /* RdCost.cpp:73-78 */
  return (uint64_t)( motionLambda * orc_mv_bits( x, y, predHor, predVer, costScale, imvShift ) );
}

/* Full search replay (EncoderLib/InterSearch.cpp:2209-2251): raster order, first strictly smaller wins.
 * blk[i] = { x, y, w, h, left, right, top, bottom, predHor, predVer }; out[i] = { dx, dy, cost lo, cost hi } */
void orc_full_search( const Pel* orgPlane, int so, const Pel* refPlane, int sr, const int32_t* blk, int n, int subShift, double lambda,
                      int costScale, int imvShift, int32_t* out, uint32_t* sadTables, int tableStride )
{
  for( int i = 0; i < n; i++ )
  {
    const int32_t* d = blk + 10 * (size_t) i;
    const Pel* org = orgPlane + (ptrdiff_t) d[1] * so + d[0];
    uint64_t best = UINT64_MAX; int bx = 0, by = 0, k = 0;
    for( int dy = d[6]; dy <= d[7]; dy++ )
      for( int dx = d[4]; dx <= d[5]; dx++, k++ )
      {
        uint64_t c = orc_sad( org, so, refPlane + (ptrdiff_t)( d[1] + dy ) * sr + d[0] + dx, sr, d[2], d[3], subShift );
        if( sadTables ) sadTables[(size_t) i * tableStride + k] = (uint32_t) c;
        c += orc_mv_cost( lambda, dx, dy, d[8], d[9], costScale, imvShift );
        if( c < best ) { best = c; bx = dx; by = dy; }
      }
    out[4 * i] = bx; out[4 * i + 1] = by; out[4 * i + 2] = (int32_t)( best & 0xffffffffu ); out[4 * i + 3] = (int32_t)( best >> 32 );
  }
}

/* ------------------------------------------------------------------------------------------------------
 * Forward 2-D transform (CommonLib/TrQuant.cpp:481-564 xT; TrQuant_EMT.cpp:366-421 _fastForwardMM and the
 * B2/B4 butterflies :197-300,1106,1507 which equal the matrix product).  trHor/trVer: 0 DCT2, 1 DCT8, 2 DST7.
 * ---------------------------------------------------------------------------------------------------- */
static const int8_t* tr_matrix( int type, int N )
{
  const int off = vvc_tr_offset_host[type][ilog2u( N )];
  return off < 0 ? NULL : vvc_tr_table_host + off;
}

int orc_fwd_transform( int trHor, int trVer, const Pel* resi, int stride, int w, int h, int bitDepth, int32_t* coef )
{
  const int8_t* th = tr_matrix( trHor, w );
  const int8_t* tv = tr_matrix( trVer, h );
  if( !th || !tv ) return -1;
  const int skipW = ( trHor != 0 && w == 32 ) ? 16 : ( w > 32 ? w - 32 : 0 );    /* TrQuant.cpp:496-497 */
  const int skipH = ( trVer != 0 && h == 32 ) ? 16 : ( h > 32 ? h - 32 : 0 );
  const int s1 = ilog2u( w ) + bitDepth + 6 - 15;                                 /* :544 */
  const int s2 = ilog2u( h ) + 6;                                                 /* :545 */
  const int keepW = w - skipW, keepH = h - skipH;
  int32_t* tmp = (int32_t*) malloc( sizeof( int32_t ) * w * h );
  /* stage 1: tmp[j*h + i] = (sum_k resi[i][k] * Th[j][k] + rnd) >> s1, j < keepW  (stored transposed, 'line' = h) */
  const int r1 = s1 > 0 ? 1 << ( s1 - 1 ) : 0;
  for( int i = 0; i < h; i++ )
    for( int j = 0; j < keepW; j++ )
    {
      int32_t sum = 0;
      for( int k = 0; k < w; k++ ) sum += resi[i * stride + k] * th[j * w + k];
      tmp[j * h + i] = ( sum + r1 ) >> s1;
    }
  /* stage 2: coef[j*w + i] = (sum_k tmp[i][k] * Tv[j][k] + rnd) >> s2 over i < keepW lines, j < keepH */
  memset( coef, 0, sizeof( int32_t ) * w * h );
  const int r2 = 1 << ( s2 - 1 );
  for( int i = 0; i < keepW; i++ )
    for( int j = 0; j < keepH; j++ )
    {
      int32_t sum = 0;
      for( int k = 0; k < h; k++ ) sum += tmp[i * h + k] * tv[j * h + k];
      coef[j * w + i] = ( sum + r2 ) >> s2;
    }
  free( tmp );
  return 0;
}

/* bare 1-D core as unit-tested by the reference (TrQuant_EMT.cpp:1973-2000 fastFwdCore) */
void orc_fwd_core( int trSize, const int16_t* tc, const int32_t* src, int32_t* dst, unsigned line, unsigned reducedLine, unsigned cutoff, int shift )
{
  const int rnd = 1 << ( shift - 1 );
  for( unsigned i = 0; i < reducedLine; i++ )
    for( unsigned j = 0; j < cutoff; j++ )
    {
      int32_t sum = 0;
      for( int k = 0; k < trSize; k++ ) sum += src[i * trSize + k] * tc[j * trSize + k];
      dst[j * line + i] = ( sum + rnd ) >> shift;
    }
}

/* ------------------------------------------------------------------------------------------------------
 * Coefficient scan (CommonLib/Rom.cpp:1098-1136 ScanGenerator, :1236-1284 grouped 4x4 up-right diagonal)
 * for blocks with w,h >= 4: groups of 4x4 inside the min(32,w) x min(32,h) region.
 * ---------------------------------------------------------------------------------------------------- */
static void diag_scan( int bw, int bh, int* xs, int* ys )
{
  int line = 0, col = 0;
  for( int i = 0; i < bw * bh; i++ )
  {
    xs[i] = col; ys[i] = line;
    if( col == bw - 1 || line == 0 )
    {
      line += col + 1; col = 0;
      if( line >= bh ) { col += line - ( bh - 1 ); line = bh - 1; }
    }
    else { col++; line--; }
  }
}

int orc_scan_order( int w, int h, int32_t* idx )
{
  const int gw = ( w < 32 ? w : 32 ) >> 2, gh = ( h < 32 ? h : 32 ) >> 2;
  int gx[64], gy[64], cx[16], cy[16];
  diag_scan( gw, gh, gx, gy );
  diag_scan( 4, 4, cx, cy );
  for( int g = 0; g < gw * gh; g++ )
    for( int c = 0; c < 16; c++ )
      idx[g * 16 + c] = ( gy[g] * 4 + cy[c] ) * w + gx[g] * 4 + cx[c];
  return gw * gh * 16;
}

/* ------------------------------------------------------------------------------------------------------
 * Plain quantiser (CommonLib/Quant.cpp:132-230 QuantCore, wrapper :735-833 without sign-bit hiding).
 * Luma, no scaling lists, no LFNST, no transform skip; maxLog2TrDynamicRange = 15 (Slice.h:776).
 * qp is the CU QP (cu.qp); the quantiser uses qp + 6*(bitDepth-8) (Quant.cpp:99).
 * ---------------------------------------------------------------------------------------------------- */
typedef struct { int scale, qbits; int64_t add; } QuantPar;

static QuantPar quant_par_ex( int w, int h, int bitDepth, int qp, int addNum, int plusOne )
{
  QuantPar p;
  int baseQp = qp + 6 * ( bitDepth - 8 );
  if( baseQp < 0 ) baseQp = 0;
  if( baseQp > 63 + 6 * ( bitDepth - 8 ) ) baseQp = 63 + 6 * ( bitDepth - 8 );
  baseQp += plusOne;                                                                    /* Quant.cpp:853: cQP.Qp( false ) + 1, after QpParam's clip (:113) */
  const int per = baseQp / 6, rem = baseQp % 6;
  const int sqrt2 = ( ilog2u( w ) + ilog2u( h ) ) & 1;                                  /* UnitTools.cpp:3616 */
  const int trShift = 15 - bitDepth - ( ( ilog2u( w ) + ilog2u( h ) ) >> 1 ) - sqrt2;   /* Quant.h:69-72 */
  p.scale = vvc_quant_scales_host[sqrt2][rem];
  p.qbits = 14 + per + trShift;                                                         /* Quant.cpp:769 */
  p.add   = (int64_t) addNum << ( p.qbits - 9 );
  return p;
}
static QuantPar quant_par( int w, int h, int bitDepth, int qp, int addNum ) { return quant_par_ex( w, h, bitDepth, qp, addNum, 0 ); }

/* Sign-bit hiding of the plain quantiser: Quant::xSignBitHidingHDQ (CommonLib/Quant.cpp:377-518), run by Quant::quant when the slice enables sign data
 * hiding and absSum >= 2 (:817-826).  Per coefficient group (from the one holding the last level down to the first): if the distance between the first and the
 * last non-zero level is at least SBH_THRESHOLD = 4 (CommonDef.h:272) and the parity of the level sum differs from the sign of the first non-zero level, the level
 * whose change costs least -- judged by deltaU, the quantisation remainder QuantCore leaves (:221) -- is moved by one.  deltaU is recomputed here from the
 * coefficient (same formula); only positions QuantCore quantised are visited. */
static int32_t sbh_delta_u( int32_t c, const QuantPar* p )
{
  const int64_t t = (int64_t) iabs( c ) * p->scale;
  const int32_t mag = (int32_t)( ( t + p->add ) >> p->qbits );
  return (int32_t)( ( t - ( (int64_t) mag << p->qbits ) ) >> ( p->qbits - 8 ) );
}
static void sign_bit_hiding( int16_t* q, const int32_t* coef, const int32_t* scan, const QuantPar* p, int* lastScanPos )
{
  const int32_t cmax = 32767, cmin = -32768;                       /* entropyCoding limits for maxLog2TrDynamicRange = 15 */
  int lastCG = -1;
  for( int subSet = *lastScanPos >> 4; subSet >= 0; subSet-- )
  {
    const int subPos = subSet << 4;
    int firstNZ = 16, lastNZ = -1, absSum = 0, n;
    for( n = 15; n >= 0; n-- ) if( q[scan[n + subPos]] ) { lastNZ = n; break; }
    for( n = 0; n < 16; n++ )  if( q[scan[n + subPos]] ) { firstNZ = n; break; }
    for( n = firstNZ; n <= lastNZ; n++ ) absSum += q[scan[n + subPos]];
    if( lastNZ >= 0 && lastCG == -1 ) lastCG = 1;
    if( lastNZ - firstNZ >= 4 )
    {
      const uint32_t signbit = q[scan[subPos + firstNZ]] > 0 ? 0 : 1;
      if( signbit != ( (uint32_t) absSum & 1u ) )
      {
        int32_t curCost = INT32_MAX, minCostInc = INT32_MAX;
        int minPos = -1, finalChange = 0, curChange = 0, minScanPos = -1;
        for( n = ( lastCG == 1 ? lastNZ : 15 ); n >= 0; --n )
        {
          const int blkPos = scan[n + subPos];
          const int32_t dU = sbh_delta_u( coef[blkPos], p );
          if( q[blkPos] != 0 )
          {
            if( dU > 0 ) { curCost = -dU; curChange = 1; }
            else if( n == firstNZ && iabs( q[blkPos] ) == 1 ) curCost = INT32_MAX;
            else { curCost = dU; curChange = -1; }
          }
          else if( n < firstNZ )
          {
            const uint32_t thisSign = coef[blkPos] >= 0 ? 0 : 1;
            if( thisSign != signbit ) curCost = INT32_MAX;
            else { curCost = -dU; curChange = 1; }
          }
          else { curCost = -dU; curChange = 1; }
          if( curCost < minCostInc ) { minCostInc = curCost; finalChange = curChange; minPos = blkPos; minScanPos = n + subPos; }
        }
        if( q[minPos] == cmax || q[minPos] == cmin ) finalChange = -1;
        if( coef[minPos] >= 0 ) q[minPos] = (int16_t)( q[minPos] + finalChange ); else q[minPos] = (int16_t)( q[minPos] - finalChange );
        if( minScanPos == *lastScanPos && q[minPos] == 0 )
          for( ; *lastScanPos >= 0 && q[scan[*lastScanPos]] == 0; ( *lastScanPos )-- );
        else if( minScanPos > *lastScanPos && q[minPos] != 0 ) *lastScanPos = minPos;     /* sic: block position, as the reference writes it (:508) */
      }
    }
    if( lastCG == 1 ) lastCG = 0;
  }
}

int orc_quant_ex( const int32_t* coef, int w, int h, int bitDepth, int qp, int isIRAP, int signHiding, int16_t* q, int32_t* absSum, int32_t* lastPos );
int orc_quant( const int32_t* coef, int w, int h, int bitDepth, int qp, int isIRAP, int16_t* q, int32_t* absSum, int32_t* lastPos )
{
  return orc_quant_ex( coef, w, h, bitDepth, qp, isIRAP, 0, q, absSum, lastPos );
}

static int quant_core( const int32_t* coef, int w, int h, QuantPar p, int signHiding, int16_t* q, int32_t* absSum, int32_t* lastPos )
{
  int32_t scan[1024];
  const int nScan = orc_scan_order( w, h, scan );
  int pos = nScan - 1;
  for( ; pos > 0; pos-- ) if( coef[scan[pos]] ) break;                                 /* :160-165 */
  const int thrVal = 8;                                                                /* vvencCfg.cpp:971-973 */
  const int32_t thres = p.qbits ? (int32_t)( (int64_t) thrVal << ( p.qbits - 1 ) ) : (int32_t)( (int64_t)( thrVal >> 1 ) << p.qbits );
  const int32_t useThres = thres / ( p.scale << 2 );                                   /* :180 */
  for( int sub = pos >> 4; sub >= 1; sub-- )                                           /* :184-208 */
  {
    if( pos >= 16 )
    {
      const int inCg = pos & 15;
      int allSmaller = 1;
      for( int k = inCg, sp = pos; allSmaller && k >= 0; k--, sp-- ) allSmaller &= iabs( coef[scan[sp]] ) <= useThres;
      if( allSmaller ) { pos -= inCg + 1; continue; }
      else break;
    }
  }
  memset( q, 0, sizeof( int16_t ) * w * h );
  int32_t sum = 0;
  for( int cp = 0; cp <= pos; cp++ )
  {
    const int32_t c = coef[scan[cp]];
    const int64_t t = (int64_t) iabs( c ) * p.scale;
    const int32_t mag = (int32_t)( ( t + p.add ) >> p.qbits );
    sum += mag;
    int32_t v = c < 0 ? -mag : mag;
    if( v < -32768 ) v = -32768; if( v > 32767 ) v = 32767;
    q[scan[cp]] = (int16_t) v;
  }
  int last = pos;
  if( sum )                                                                            /* Quant.cpp:806-816 */
    for( int sp = pos; sp >= 0; sp-- ) if( q[scan[sp]] ) { last = sp; break; }
  if( sum >= 2 && signHiding ) sign_bit_hiding( q, coef, scan, &p, &last );            /* Quant.cpp:817-826 */
  *absSum = sum; *lastPos = last;
  return 0;
}

int orc_quant_ex( const int32_t* coef, int w, int h, int bitDepth, int qp, int isIRAP, int signHiding, int16_t* q, int32_t* absSum, int32_t* lastPos )
{
  return quant_core( coef, w, h, quant_par( w, h, bitDepth, qp, isIRAP ? 171 : 85 ), signHiding, q, absSum, lastPos );               /* Quant.cpp:772 */
}

/* ------------------------------------------------------------------------------------------------------
 * Transform skip (tu.mtsIdx == MTS_SKIP): TrQuant::xTransformSkip copies the residual into the coefficient buffer (TrQuant.cpp:1050-1064), Quant::quant runs with
 * cQP.per / rem( true ) -- the QP raised to 4 + 6 * internalMinusInputBitDepth (Quant.cpp:117-124) --, no transform shift in iQBits (:772) and the first row of
 * g_quantScales (TU::needsSqrt2Scale is false for skipped transforms); Quant::dequant drops the transform shift likewise (:561) and xITransformSkip casts the
 * dequantised coefficient to Pel (:659-675).  xNeedRDOQ keeps the transform shift in its own iQBits even for skipped transforms (:868-873) and uses 256 instead of
 * 171 for chroma components (:877).  inputDelta = sps.internalMinusInputBitDepth.
 * ---------------------------------------------------------------------------------------------------- */
static int ts_base_qp( int bitDepth, int qp, int inputDelta )
{
  int baseQp = qp + 6 * ( bitDepth - 8 );
  if( baseQp < 0 ) baseQp = 0;
  if( baseQp > 63 + 6 * ( bitDepth - 8 ) ) baseQp = 63 + 6 * ( bitDepth - 8 );
  const int minTs = 4 + 6 * inputDelta;
  return baseQp > minTs ? baseQp : minTs;
}
int orc_quant_ts( const int32_t* coef, int w, int h, int bitDepth, int qp, int isIRAP, int signHiding, int inputDelta, int16_t* q, int32_t* absSum, int32_t* lastPos )
{
  const int baseQp = ts_base_qp( bitDepth, qp, inputDelta );
  QuantPar p;
  p.scale = vvc_quant_scales_host[0][baseQp % 6];
  p.qbits = 14 + baseQp / 6;
  p.add   = (int64_t)( isIRAP ? 171 : 85 ) << ( p.qbits - 9 );
  return quant_core( coef, w, h, p, signHiding, q, absSum, lastPos );
}
int orc_transform_quant_ts( const Pel* resi, int stride, int w, int h, int bitDepth, int qp, int isIRAP, int signHiding, int inputDelta,
                            int32_t* coef, int16_t* q, int32_t* absSum, int32_t* lastPos )
{
  if( w > 32 || h > 32 ) return -1;                                                    /* log2MaxTransformSkipBlockSize <= 5 */
  for( int y = 0; y < h; y++ ) for( int x = 0; x < w; x++ ) coef[y * w + x] = resi[y * stride + x];
  return orc_quant_ts( coef, w, h, bitDepth, qp, isIRAP, signHiding, inputDelta, q, absSum, lastPos );
}
/* Quant::xNeedRDOQ in full: depQuant only counts for non-skipped transforms; chroma components use 256 */
int orc_need_rdoq_ex( const int32_t* coef, int w, int h, int bitDepth, int qp, int depQuant, int transformSkip, int inputDelta, int chroma )
{
  int baseQp;
  if( transformSkip ) baseQp = ts_base_qp( bitDepth, qp, inputDelta );
  else
  {
    baseQp = qp + 6 * ( bitDepth - 8 );
    if( baseQp < 0 ) baseQp = 0;
    if( baseQp > 63 + 6 * ( bitDepth - 8 ) ) baseQp = 63 + 6 * ( bitDepth - 8 );
    if( depQuant ) baseQp += 1;
  }
  const int sqrt2 = transformSkip ? 0 : ( ( ilog2u( w ) + ilog2u( h ) ) & 1 );
  const int trShift = 15 - bitDepth - ( ( ilog2u( w ) + ilog2u( h ) ) >> 1 ) - sqrt2;
  const int scale = vvc_quant_scales_host[sqrt2][baseQp % 6], qbits = 14 + baseQp / 6 + trShift;
  const int64_t add = (int64_t)( chroma ? 256 : 171 ) << ( qbits - 9 );
  const int n = w * ( h < 32 ? h : 32 );
  for( int i = 0; i < n; i++ )
  {
    const int64_t t = (int64_t) iabs( coef[i] ) * scale;
    if( (int32_t)( ( t + add ) >> qbits ) != 0 ) return 1;
  }
  return 0;
}


/* ------------------------------------------------------------------------------------------------------
 * LFNST, forward (SURVEY 8f-4): TrQuant::xFwdLfnst (CommonLib/TrQuant.cpp:942-1048) with xFwdLfnstNxNCore (:166-187) between TrQuant::xT and the quantiser.
 * The primary transform keeps only the top-left 4x4 (a 4-pel side) or 8x8 region when the CU carries an LFNST index (:499-511); its first 16 resp. 48
 * coefficients (rows of 8 then rows of 4, or the transposed walk) go through a 16x16 / 16x48 int8 kernel chosen by (set = g_lfnstLut[intra mode], index),
 * (sum + 64) >> 7, only the first 8 (4x4 and 8x8 TUs) or 16 outputs are kept, and the outputs land on the first scan positions of the top-left region
 * (g_coefTopLeftDiagScan8x8 / the TU's grouped scan).  The quantiser then only looks at coefficient group 0 (Quant.cpp:151-158).
 * set (0..3), index (1..2) and transpose come from the host: they follow from the intra mode through the reference's own xGetLFNSTIntraMode / g_lfnstLut /
 * xGetTransposeFlag.
 * ---------------------------------------------------------------------------------------------------- */
void orc_fwd_lfnst( int32_t* coef, int w, int h, int set, int lfnstIdx, int transpose )
{
  const int whge3 = w >= 8 && h >= 8, sb = whge3 ? 8 : 4, nIn = whge3 ? 48 : 16;
  const int zeroOut = ( ( w == 4 && h == 4 ) || ( w == 8 && h == 8 ) ) ? 8 : 16;
  const int8_t* mat = (const int8_t*) vvc_lfnst_words + ( whge3 ? ( set * 2 + ( lfnstIdx - 1 ) ) * 16 * 48 : VVC_LFNST_4X4_OFFSET + ( set * 2 + ( lfnstIdx - 1 ) ) * 16 * 16 );
  int32_t in[48], out[48];
  for( int i = 0; i < nIn; i++ )
  {
    int a, b;                                  /* a: index along the walk's fast axis, b: slow axis */
    if( sb == 4 ) { b = i >> 2; a = i & 3; }
    else if( i < 32 ) { b = i >> 3; a = i & 7; }
    else { b = 4 + ( ( i - 32 ) >> 2 ); a = ( i - 32 ) & 3; }
    const int x = transpose ? b : a, y = transpose ? a : b;           /* :973-1019 */
    in[i] = coef[y * w + x];
  }
  for( int j = 0; j < nIn; j++ )
  {
    if( j < zeroOut )
    {
      int32_t sum = 0;
      for( int i = 0; i < nIn; i++ ) sum += in[i] * mat[j * nIn + i];
      out[j] = ( sum + 64 ) >> 7;
    }
    else out[j] = 0;                            /* :185 memset */
  }
  /* forward spectral rearrangement (:1037-1046): grouped 4x4 diagonal scan of the top-left region, groups (0,0), (0,1), (1,0) */
  int gx[4], gy[4], cx[16], cy[16];
  diag_scan( 2, 2, gx, gy ); diag_scan( 4, 4, cx, cy );
  for( int j = 0; j < nIn; j++ )
  {
    const int g = j >> 4, c = j & 15;
    coef[( gy[g] * 4 + cy[c] ) * w + gx[g] * 4 + cx[c]] = out[j];
  }
}

/* TrQuant::transformNxN for a luma TU of an intra CU with cu.lfnstIdx = lfnstIdx (1..2): xT with the LFNST zero-out, xFwdLfnst, Quant::quant (plain quantiser,
 * optional sign-bit hiding) and xNeedRDOQ on the same coefficients.  Transform types are DCT-II (LFNST and MTS exclude each other, IntraSearch). */
int orc_transform_quant_lfnst( const Pel* resi, int stride, int w, int h, int bitDepth, int qp, int isIRAP, int signHiding, int set, int lfnstIdx, int transpose,
                               int32_t* coef, int16_t* q, int32_t* absSum, int32_t* lastPos )
{
  if( orc_fwd_transform( 0, 0, resi, stride, w, h, bitDepth, coef ) ) return -1;
  const int keep = ( w >= 8 && h >= 8 ) ? 8 : 4;                                       /* TrQuant.cpp:499-511 */
  for( int y = 0; y < h; y++ ) for( int x = 0; x < w; x++ ) if( x >= keep || y >= keep ) coef[y * w + x] = 0;
  orc_fwd_lfnst( coef, w, h, set, lfnstIdx, transpose );
  const QuantPar p = quant_par( w, h, bitDepth, qp, isIRAP ? 171 : 85 );
  int32_t scan[1024];
  orc_scan_order( w, h, scan );
  int pos = ( ( w == 4 && h == 4 ) || ( w == 8 && h == 8 ) ) ? 7 : 15;                 /* Quant.cpp:151-158: one coefficient group, 8 positions for 4x4 / 8x8 */
  for( ; pos > 0; pos-- ) if( coef[scan[pos]] ) break;
  memset( q, 0, sizeof( int16_t ) * w * h );
  int32_t sum = 0;
  for( int cp = 0; cp <= pos; cp++ )
  {
    const int32_t c = coef[scan[cp]];
    const int64_t t = (int64_t) iabs( c ) * p.scale;
    const int32_t mag = (int32_t)( ( t + p.add ) >> p.qbits );
    sum += mag;
    int32_t v = c < 0 ? -mag : mag;
    if( v < -32768 ) v = -32768; if( v > 32767 ) v = 32767;
    q[scan[cp]] = (int16_t) v;
  }
  int last = pos;
  if( sum ) for( int sp = pos; sp >= 0; sp-- ) if( q[scan[sp]] ) { last = sp; break; }
  if( sum >= 2 && signHiding ) sign_bit_hiding( q, coef, scan, &p, &last );
  *absSum = sum; *lastPos = last;
  return 0;
}

/* needRdoqCore (CommonLib/Quant.cpp:264-278) through Quant::xNeedRDOQ (:835-891), luma */
int orc_need_rdoq( const int32_t* coef, int w, int h, int bitDepth, int qp, int depQuant )
{
  const QuantPar p = quant_par_ex( w, h, bitDepth, qp, 171, depQuant ? 1 : 0 );
  const int n = w * ( h < 32 ? h : 32 );
  for( int i = 0; i < n; i++ )
  {
    const int64_t t = (int64_t) iabs( coef[i] ) * p.scale;
    if( (int32_t)( ( t + p.add ) >> p.qbits ) != 0 ) return 1;
  }
  return 0;
}

int orc_transform_quant( int trHor, int trVer, const Pel* resi, int stride, int w, int h, int bitDepth, int qp, int isIRAP,
                         int32_t* coef, int16_t* q, int32_t* absSum, int32_t* lastPos )
{
  if( orc_fwd_transform( trHor, trVer, resi, stride, w, h, bitDepth, coef ) ) return -1;
  return orc_quant( coef, w, h, bitDepth, qp, isIRAP, q, absSum, lastPos );
}
/* list form over the blocks of two planes: TU i takes the residual org(x, y) - ref(x + dx, y + dy) of pos[i] = { x, y, dx, dy }, then
 * orc_transform_quant and orc_need_rdoq on its coefficients; q holds n compact w x h level blocks */
int orc_transform_quant_blocks( int trHor, int trVer, const Pel* orgPlane, int so, const Pel* refPlane, int sr, const int32_t* pos, int n, int w, int h,
                                int bitDepth, int qp, int isIRAP, int depQuant, int16_t* q, int32_t* absSum, int32_t* lastPos, uint8_t* needRdoq )
{
  Pel* resi = (Pel*) malloc( sizeof( Pel ) * w * h );
  int32_t* coef = (int32_t*) malloc( sizeof( int32_t ) * w * h );
  int rc = 0;
  for( int i = 0; i < n && !rc; i++ )
  {
    const int32_t* d = pos + 4 * (size_t) i;
    const Pel* o = orgPlane + (ptrdiff_t) d[1] * so + d[0];
    const Pel* r = refPlane + (ptrdiff_t)( d[1] + d[3] ) * sr + d[0] + d[2];
    for( int y = 0; y < h; y++ )
      for( int x = 0; x < w; x++ ) resi[y * w + x] = (Pel)( o[y * so + x] - r[y * sr + x] );
    rc = orc_transform_quant( trHor, trVer, resi, w, w, h, bitDepth, qp, isIRAP, coef, q + (size_t) i * w * h, absSum + i, lastPos + i );
    needRdoq[i] = (uint8_t) orc_need_rdoq( coef, w, h, bitDepth, qp, depQuant );
  }
  free( resi ); free( coef );
  return rc;
}

/* same with slice->signDataHidingEnabled (Quant.cpp:748) */
int orc_transform_quant_ex( int trHor, int trVer, const Pel* resi, int stride, int w, int h, int bitDepth, int qp, int isIRAP, int signHiding,
                            int32_t* coef, int16_t* q, int32_t* absSum, int32_t* lastPos )
{
  if( orc_fwd_transform( trHor, trVer, resi, stride, w, h, bitDepth, coef ) ) return -1;
  return orc_quant_ex( coef, w, h, bitDepth, qp, isIRAP, signHiding, q, absSum, lastPos );
}

/* ------------------------------------------------------------------------------------------------------
 * Inverse path of the TU loop (SURVEY 8f rank 1): Quant::dequant (CommonLib/Quant.cpp:520-609) with DeQuantCore
 * (:232-262), TrQuant::xIT (CommonLib/TrQuant.cpp:567-660) with _fastInverseMM / the B2..B8 butterflies which equal the
 * matrix product (TrQuant_EMT.cpp:64-194,231-636), PelBuf::reconstruct (Buffer.cpp:719) and the SSE that follows
 * (IntraSearch.cpp:1353-1429, InterSearch.cpp:3659-3714).  Luma, no scaling lists / LFNST / transform skip / BDPCM.
 * ---------------------------------------------------------------------------------------------------- */
static const int inv_quant_scales[2][6] = { { 40, 45, 51, 57, 64, 72 }, { 57, 64, 72, 80, 90, 102 } };   /* Rom.cpp:1396-1400 */

static inline int32_t clip3i( int32_t lo, int32_t hi, int32_t v ) { return v < lo ? lo : ( v > hi ? hi : v ); }

int orc_dequant( const int16_t* q, int w, int h, int bitDepth, int qp, int32_t* coef )
{
  int baseQp = qp + 6 * ( bitDepth - 8 );
  if( baseQp < 0 ) baseQp = 0;
  if( baseQp > 63 + 6 * ( bitDepth - 8 ) ) baseQp = 63 + 6 * ( bitDepth - 8 );
  const int per = baseQp / 6, rem = baseQp % 6;
  const int sqrt2 = ( ilog2u( w ) + ilog2u( h ) ) & 1;
  const int trShift = 15 - bitDepth - ( ( ilog2u( w ) + ilog2u( h ) ) >> 1 ) - sqrt2;    /* Quant.cpp:554-556 */
  const int rightShift = 6 - ( trShift + per );                                          /* :561, IQUANT_SHIFT = 6 */
  const int scale = inv_quant_scales[sqrt2][rem];
  int tib = 32 + rightShift - 7; if( tib > 16 ) tib = 16;                                /* :606 targetInputBitDepth */
  const int32_t inMax = ( 1 << ( tib - 1 ) ) - 1, inMin = -( inMax + 1 );
  const int32_t trMax = 32767, trMin = -32768;
  for( int n = 0; n < w * h; n++ )
  {
    const int32_t c = clip3i( inMin, inMax, q[n] );
    int32_t v;
    if( rightShift > 0 ) v = ( c * scale + ( 1 << ( rightShift - 1 ) ) ) >> rightShift;   /* :238-249 */
    else                 v = (int32_t)( (uint32_t)( c * scale ) << ( -rightShift ) );     /* :251-261 (int32 product times 2^leftShift) */
    coef[n] = clip3i( trMin, trMax, v );
  }
  return 0;
}

int orc_inv_transform( int trHor, int trVer, const int32_t* coef, int w, int h, int bitDepth, Pel* resi, int stride );
/* Dequantiser of dependent quantisation: DQIntern::Quantizer::dequantBlock (CommonLib/DepQuant.cpp:574-629), what DepQuant::dequant runs for non-skipped transforms of
 * a slice with depQuantEnabled.  Walks the scan from the last significant position down with the 4-state machine (state' = (32040 >> ((state << 2) + ((level & 1) << 1))) & 3);
 * a level reconstructs from qIdx = 2 * level -+ (state >> 1) at QP + 1.  Positions above the last significant one hold zero levels, which keep state 0, so the walk may
 * start at the end of the scan.  No scaling lists. */
int orc_dequant_dq( const int16_t* q, int w, int h, int bitDepth, int qp, int32_t* coef )
{
  int baseQp = qp + 6 * ( bitDepth - 8 );
  if( baseQp < 0 ) baseQp = 0;
  if( baseQp > 63 + 6 * ( bitDepth - 8 ) ) baseQp = 63 + 6 * ( bitDepth - 8 );
  const int qpDQ = baseQp + 1, per = qpDQ / 6, rem = qpDQ - 6 * per;
  const int sqrt2 = ( ilog2u( w ) + ilog2u( h ) ) & 1;
  const int trShift = 15 - bitDepth - ( ( ilog2u( w ) + ilog2u( h ) ) >> 1 ) - sqrt2;
  const int shift = 6 + 1 - per - trShift;                                               /* :607 */
  int32_t scale = inv_quant_scales[sqrt2][rem];
  const int32_t add = shift < 0 ? 0 : ( ( 1 << shift ) >> 1 );
  if( shift < 0 ) scale <<= -shift;                                                      /* :619-622: applied once, at the last position, and kept */
  int32_t scan[1024];
  const int nScan = orc_scan_order( w, h, scan );
  memset( coef, 0, sizeof( int32_t ) * w * h );
  int state = 0;
  for( int sp = nScan - 1; sp >= 0; sp-- )
  {
    const int32_t level = q[scan[sp]];
    if( level )
    {
      const int32_t qIdx = 2 * level + ( level > 0 ? -( state >> 1 ) : ( state >> 1 ) );
      const int64_t nom = ( (int64_t) qIdx * scale + add ) >> ( shift < 0 ? 0 : shift );
      coef[scan[sp]] = (int32_t)( nom < -32768 ? -32768 : ( nom > 32767 ? 32767 : nom ) );
    }
    state = ( 32040 >> ( ( state << 2 ) + ( ( level & 1 ) << 1 ) ) ) & 3;
  }
  return 0;
}
int orc_inv_transform_quant_dq( int trHor, int trVer, const int16_t* q, int w, int h, int bitDepth, int qp, int32_t* coef, Pel* resi, int stride )
{
  orc_dequant_dq( q, w, h, bitDepth, qp, coef );
  return orc_inv_transform( trHor, trVer, coef, w, h, bitDepth, resi, stride );
}

/* xIT: first pass over columns (vertical transform, shift 7), second over rows (shift 20 - bitDepth); both clip to 16 bit */
int orc_inv_transform( int trHor, int trVer, const int32_t* coef, int w, int h, int bitDepth, Pel* resi, int stride )
{
  const int8_t* th = tr_matrix( trHor, w );
  const int8_t* tv = tr_matrix( trVer, h );
  if( !th || !tv ) return -1;
  const int skipW = ( trHor != 0 && w == 32 ) ? 16 : ( w > 32 ? w - 32 : 0 );    /* TrQuant.cpp:588-589 */
  const int skipH = ( trVer != 0 && h == 32 ) ? 16 : ( h > 32 ? h - 32 : 0 );
  const int s1 = 7, s2 = 20 - bitDepth;                                          /* :608-609 */
  int32_t* tmp = (int32_t*) calloc( (size_t) w * h, sizeof( int32_t ) );
  /* pass 1 (fastInvTrans[trVer], line = w, skip lines = skipW, cutoff = h - skipH): tmp[i*h + j] = clip((sum_k coef[k*w + i] * Tv[k][j] + 64) >> 7) */
  for( int i = 0; i < w - skipW; i++ )
    for( int j = 0; j < h; j++ )
    {
      int32_t sum = 0;
      for( int k = 0; k < h - skipH; k++ ) sum += coef[k * w + i] * tv[k * h + j];
      tmp[i * h + j] = clip3i( -32768, 32767, ( sum + ( 1 << ( s1 - 1 ) ) ) >> s1 );
    }
  /* pass 2 (fastInvTrans[trHor], line = h, no skipped lines, cutoff = w - skipW): blk[i*w + j] = clip((sum_k tmp[k*h + i] * Th[k][j] + rnd) >> s2) */
  for( int i = 0; i < h; i++ )
    for( int j = 0; j < w; j++ )
    {
      int32_t sum = 0;
      for( int k = 0; k < w - skipW; k++ ) sum += tmp[k * h + i] * th[k * w + j];
      resi[i * stride + j] = (Pel) clip3i( -32768, 32767, ( sum + ( 1 << ( s2 - 1 ) ) ) >> s2 );
    }
  free( tmp );
  return 0;
}

/* TrQuant::invTransformNxN (TrQuant.cpp:318-348) */
int orc_inv_transform_quant( int trHor, int trVer, const int16_t* q, int w, int h, int bitDepth, int qp, int32_t* coef, Pel* resi, int stride )
{
  orc_dequant( q, w, h, bitDepth, qp, coef );
  return orc_inv_transform( trHor, trVer, coef, w, h, bitDepth, resi, stride );
}

/* the same for a skipped transform: dequant without the transform shift, residual = Pel( coefficient ) */
int orc_inv_transform_quant_ts( const int16_t* q, int w, int h, int bitDepth, int qp, int inputDelta, int32_t* coef, Pel* resi, int stride )
{
  const int baseQp = ts_base_qp( bitDepth, qp, inputDelta );
  const int per = baseQp / 6, rem = baseQp % 6;
  const int rightShift = 6 - per;                                                        /* Quant.cpp:561 with isTransformSkip */
  const int scale = inv_quant_scales[0][rem];
  int tib = 32 + rightShift - 7; if( tib > 16 ) tib = 16;
  const int32_t inMax = ( 1 << ( tib - 1 ) ) - 1, inMin = -( inMax + 1 );
  for( int n = 0; n < w * h; n++ )
  {
    const int32_t c = clip3i( inMin, inMax, q[n] );
    int32_t v;
    if( rightShift > 0 ) v = ( c * scale + ( 1 << ( rightShift - 1 ) ) ) >> rightShift;
    else                 v = (int32_t)( (uint32_t)( c * scale ) << ( -rightShift ) );
    coef[n] = clip3i( -32768, 32767, v );
  }
  for( int y = 0; y < h; y++ ) for( int x = 0; x < w; x++ ) resi[y * stride + x] = (Pel) coef[y * w + x];
  return 0;
}

/* LFNST, inverse: TrQuant::xInvLfnst (TrQuant.cpp:838-940) with xInvLfnstNxNCore (:190-213) between the dequantiser and xIT.  The first 16 scan positions (the top-left
 * 4x4 group in diagonal order) hold the secondary coefficients; the inverse kernel is the transpose of the forward one (g_lfnstInv* == g_lfnstFwd*^T, checked when the
 * tables were generated), outputs are clipped to 16 bit and land on the walk the forward side read (rows of 8 then rows of 4, or transposed).  xIT then only uses the
 * top-left 8x8 (4x4) coefficients (:590-602 skipWidth / skipHeight). */
void orc_inv_lfnst( int32_t* coef, int w, int h, int set, int lfnstIdx, int transpose )
{
  const int whge3 = w >= 8 && h >= 8, sb = whge3 ? 8 : 4, nOut = whge3 ? 48 : 16;
  const int zeroOut = ( ( w == 4 && h == 4 ) || ( w == 8 && h == 8 ) ) ? 8 : 16;
  const int8_t* mat = (const int8_t*) vvc_lfnst_words + ( whge3 ? ( set * 2 + ( lfnstIdx - 1 ) ) * 16 * 48 : VVC_LFNST_4X4_OFFSET + ( set * 2 + ( lfnstIdx - 1 ) ) * 16 * 16 );
  int cx[16], cy[16];
  diag_scan( 4, 4, cx, cy );
  int32_t src[16], out[48];
  for( int i = 0; i < 16; i++ ) src[i] = coef[cy[i] * w + cx[i]];
  for( int j = 0; j < nOut; j++ )
  {
    int32_t sum = 0;
    for( int i = 0; i < zeroOut; i++ ) sum += src[i] * mat[i * nOut + j];
    out[j] = clip3i( -32768, 32767, ( sum + 64 ) >> 7 );
  }
  for( int j = 0; j < nOut; j++ )
  {
    int a, b;
    if( sb == 4 ) { b = j >> 2; a = j & 3; }
    else if( j < 32 ) { b = j >> 3; a = j & 7; }
    else { b = 4 + ( ( j - 32 ) >> 2 ); a = ( j - 32 ) & 3; }
    const int x = transpose ? b : a, y = transpose ? a : b;
    coef[y * w + x] = out[j];
  }
}
int orc_inv_transform_quant_lfnst( const int16_t* q, int w, int h, int bitDepth, int qp, int depQuant, int set, int lfnstIdx, int transpose, int32_t* coef, Pel* resi, int stride )
{
  if( depQuant ) orc_dequant_dq( q, w, h, bitDepth, qp, coef );
  else           orc_dequant( q, w, h, bitDepth, qp, coef );
  orc_inv_lfnst( coef, w, h, set, lfnstIdx, transpose );
  const int keep = ( w >= 8 && h >= 8 ) ? 8 : 4;
  for( int y = 0; y < h; y++ ) for( int x = 0; x < w; x++ ) if( x >= keep || y >= keep ) coef[y * w + x] = 0;
  return orc_inv_transform( 0, 0, coef, w, h, bitDepth, resi, stride );
}

/* PelBuf::reconstruct (Buffer.cpp:719-760): reco = ClipPel( pred + resi ) with the default clipping range [0, 2^bd - 1] */
void orc_reconstruct( const Pel* pred, int ps, const Pel* resi, int rs, Pel* reco, int cs, int w, int h, int bitDepth )
{
  const int mx = ( 1 << bitDepth ) - 1;
  for( int y = 0; y < h; y++ )
    for( int x = 0; x < w; x++ ) reco[y * cs + x] = (Pel) clip3i( 0, mx, pred[y * ps + x] + resi[y * rs + x] );
}

/* One TU candidate end to end, as xIntraCodingTUBlock does for luma (IntraSearch.cpp:1353-1429): residual = org - pred, transformNxN, then
 * (absSum > 0 ? invTransformNxN : zero residual), reconstruct, SSE(org, reco).  Also returns the residual-domain distortions of the inter loop
 * (InterSearch.cpp:3670 zero-residual SSE, :3714 SSE(orgResi, recResi)).  out4 = { dist_reco, dist_resi, dist_zero, absSum | lastPos<<32 } */
int orc_tu_roundtrip_ex( int trHor, int trVer, const Pel* org, int so, const Pel* pred, int ps, int w, int h, int bitDepth, int qp, int isIRAP, int signHiding,
                         int16_t* q, Pel* reco, int cs, uint64_t* out4 );
int orc_tu_roundtrip( int trHor, int trVer, const Pel* org, int so, const Pel* pred, int ps, int w, int h, int bitDepth, int qp, int isIRAP,
                      int16_t* q, Pel* reco, int cs, uint64_t* out4 )
{
  return orc_tu_roundtrip_ex( trHor, trVer, org, so, pred, ps, w, h, bitDepth, qp, isIRAP, 0, q, reco, cs, out4 );
}
int orc_tu_roundtrip_ex( int trHor, int trVer, const Pel* org, int so, const Pel* pred, int ps, int w, int h, int bitDepth, int qp, int isIRAP, int signHiding,
                         int16_t* q, Pel* reco, int cs, uint64_t* out4 )
{
  Pel* resi = (Pel*) malloc( sizeof( Pel ) * w * h );
  Pel* rec  = (Pel*) malloc( sizeof( Pel ) * w * h );
  Pel* zero = (Pel*) calloc( (size_t) w * h, sizeof( Pel ) );
  int32_t* coef = (int32_t*) malloc( sizeof( int32_t ) * w * h );
  for( int y = 0; y < h; y++ ) for( int x = 0; x < w; x++ ) resi[y * w + x] = (Pel)( org[y * so + x] - pred[y * ps + x] );
  int32_t absSum = 0, lastPos = 0;
  int rc = orc_transform_quant_ex( trHor, trVer, resi, w, w, h, bitDepth, qp, isIRAP, signHiding, coef, q, &absSum, &lastPos );
  if( !rc )
  {
    if( absSum > 0 ) rc = orc_inv_transform_quant( trHor, trVer, q, w, h, bitDepth, qp, coef, rec, w );
    else memset( rec, 0, sizeof( Pel ) * w * h );
    orc_reconstruct( pred, ps, rec, w, reco, cs, w, h, bitDepth );
    out4[0] = orc_sse( org, so, reco, cs, w, h );
    out4[1] = orc_sse( resi, w, rec, w, w, h );
    out4[2] = orc_sse( zero, w, resi, w, w, h );
    out4[3] = (uint64_t)(uint32_t) absSum | ( (uint64_t)(uint32_t) lastPos << 32 );
  }
  free( resi ); free( rec ); free( zero ); free( coef );
  return rc;
}

/* ------------------------------------------------------------------------------------------------------
 * MCTF block matching (CommonLib/MCTF.cpp:122-145 int, :147-203 6-tap, :205-257 4-tap); filters :72-110
 * ---------------------------------------------------------------------------------------------------- */
static const int16_t mctf_f8[16][8] = {
  {0,0,0,64,0,0,0,0},{0,1,-3,64,4,-2,0,0},{0,1,-6,62,9,-3,1,0},{0,2,-8,60,14,-5,1,0},{0,2,-9,57,19,-7,2,0},{0,3,-10,53,24,-8,2,0},
  {0,3,-11,50,29,-9,2,0},{0,3,-11,44,35,-10,3,0},{0,1,-7,38,38,-7,1,0},{0,3,-10,35,44,-11,3,0},{0,2,-9,29,50,-11,3,0},{0,2,-8,24,53,-10,3,0},
  {0,2,-7,19,57,-9,2,0},{0,1,-5,14,60,-8,2,0},{0,1,-3,9,62,-6,1,0},{0,0,-2,4,64,-3,1,0} };
static const int16_t mctf_f4[16][4] = {
  {0,64,0,0},{-2,62,4,0},{-2,58,10,-2},{-4,56,14,-2},{-4,54,16,-2},{-6,52,20,-2},{-6,46,28,-4},{-4,42,30,-4},
  {-4,36,36,-4},{-4,30,42,-4},{-4,28,46,-6},{-2,20,52,-6},{-2,16,54,-4},{-2,14,56,-4},{-2,10,58,-2},{0,4,62,-2} };

void orc_mctf_filters( int16_t* f8, int16_t* f4 ) { memcpy( f8, mctf_f8, sizeof( mctf_f8 ) ); memcpy( f4, mctf_f4, sizeof( mctf_f4 ) ); }

int32_t orc_mctf_err_int( const Pel* org, int so, const Pel* buf, int sb, int w, int h )
{
  int32_t e = 0;
  for( int y = 0; y < h; y++ )
    for( int x = 0; x < w; x++ ) { const int d = org[y * so + x] - buf[y * sb + x]; e += d * d; }
  return e;
}

int32_t orc_mctf_err_frac( int tap4, const Pel* org, int so, const Pel* buf, int sb, int w, int h, int fx, int fy, int bitDepth )
{
  const int maxv = ( 1 << bitDepth ) - 1;
  const int taps = tap4 ? 4 : 6, first = tap4 ? 0 : 1, back = tap4 ? 1 : 2;   /* 6-tap uses entries 1..6 around x-3+1 */
  const int16_t* xf = tap4 ? mctf_f4[fx] : mctf_f8[fx];
  const int16_t* yf = tap4 ? mctf_f4[fy] : mctf_f8[fy];
  int32_t e = 0;
  int tmp[( 64 + 8 ) * 64];
  const int rows = h + taps - 1;
  for( int r = 0; r < rows; r++ )
    for( int x = 0; x < w; x++ )
    {
      int sum = 0;
      for( int t = 0; t < taps; t++ ) sum += xf[first + t] * buf[( r - back ) * sb + x - back + t];
      sum = ( sum + 32 ) >> 6;
      tmp[r * 64 + x] = sum < 0 ? 0 : ( sum > maxv ? maxv : sum );
    }
  for( int y = 0; y < h; y++ )
    for( int x = 0; x < w; x++ )
    {
      int sum = 0;
      for( int t = 0; t < taps; t++ ) sum += yf[first + t] * tmp[( y + t ) * 64 + x];
      sum = ( sum + 32 ) >> 6;
      sum = sum < 0 ? 0 : ( sum > maxv ? maxv : sum );
      const int d = sum - org[y * so + x];
      e += d * d;
    }
  return e;
}

/* MCTF::motionErrorLuma dispatch (CommonLib/MCTF.cpp:1099-1164); desc[i] = { x, y, mvx, mvy (1/16 pel), w, h } */
void orc_mctf_err_list( int tap4, const Pel* orgPlane, int so, const Pel* bufPlane, int sb, const int32_t* desc, int n, int bitDepth, int32_t* out )
{
  for( int i = 0; i < n; i++ )
  {
    const int32_t* d = desc + 6 * (size_t) i;
    int dx = d[2], dy = d[3];
    const int fx = dx & 15, fy = dy & 15;
    const Pel* org = orgPlane + (ptrdiff_t) d[1] * so + d[0];
    if( ( fx | fy ) == 0 )
    {
      dx /= 16; dy /= 16;
      out[i] = orc_mctf_err_int( org, so, bufPlane + (ptrdiff_t)( d[1] + dy ) * sb + d[0] + dx, sb, d[4], d[5] );
    }
    else
    {
      dx >>= 4; dy >>= 4;
      out[i] = orc_mctf_err_frac( tap4, org, so, bufPlane + (ptrdiff_t)( d[1] + dy ) * sb + d[0] + dx, sb, d[4], d[5], fx, fy, bitDepth );
    }
  }
}

/* ------------------------------------------------------------------------------------------------------
 * MCTF apply stage (SURVEY 8f rank 3): applyFrac8Core_6Tap / _4Tap (CommonLib/MCTF.cpp:259-357), applyPlanarCorrectionCore
 * (:372-420), applyBlockCore (:422-518), calcVarCore (:520-546) and the per-block body of MCTF::xFinalizeBlkLine (:1437-1483).
 * Float arithmetic follows the C++ expression types of the reference literally (float *= double rounds through double, etc.).
 * ---------------------------------------------------------------------------------------------------- */
void orc_mctf_apply_frac( int tap4, const Pel* org, int so, Pel* dst, int ds, int w, int h, int fx, int fy, int bitDepth )
{
  const int maxv = ( 1 << bitDepth ) - 1;
  const int taps = tap4 ? 4 : 6, first = tap4 ? 0 : 1, back = tap4 ? 1 : 2;
  const int16_t* xf = tap4 ? mctf_f4[fx] : mctf_f8[fx];
  const int16_t* yf = tap4 ? mctf_f4[fy] : mctf_f8[fy];
  Pel* tmp = (Pel*) malloc( sizeof( Pel ) * ( h + taps ) * w );
  for( int r = 0; r < h + taps - 1; r++ )                 /* source rows y - back .. y + h + taps - 2 - back */
    for( int x = 0; x < w; x++ )
    {
      const Pel* p = org + ( r - back ) * so + x - back;
      int sum = 0;
      for( int t = 0; t < taps; t++ ) sum += xf[first + t] * p[t];
      tmp[r * w + x] = (Pel)( ( sum + 32 ) >> 6 );        /* no clipping after the first pass (:284, :344) */
    }
  for( int y = 0; y < h; y++ )
    for( int x = 0; x < w; x++ )
    {
      int sum = 0;
      for( int t = 0; t < taps; t++ ) sum += yf[first + t] * tmp[( y + t ) * w + x];
      sum = ( sum + 32 ) >> 6;
      dst[y * ds + x] = (Pel)( sum < 0 ? 0 : ( sum > maxv ? maxv : sum ) );
    }
  free( tmp );
}

void orc_mctf_planar_correction( const Pel* ref, int rs, Pel* dst, int ds, int w, int h, int bitDepth, unsigned motionError )
{
  static const int32_t xSzm[6] = { 0, 1, 20, 336, 5440, 87296 };                 /* MCTF.cpp:369 */
  const int32_t blockSize = w * h, log2Width = ilog2u( w ), maxPel = ( 1 << bitDepth ) - 1;
  const uint32_t me2 = motionError * motionError;
  const int32_t mWeight = (int32_t)( me2 < 512u ? me2 : 512u );
  const int32_t xSum = ( blockSize * ( w - 1 ) ) >> 1;
  int32_t x1yzm = 0, x2yzm = 0, ySum = 0;
  for( int y = 0; y < h; y++ )
    for( int x = 0; x < w; x++ ) { const int32_t z = dst[y * ds + x] - ref[y * rs + x]; x1yzm += x * z; x2yzm += y * z; ySum += z; }
  const int64_t denom = (int64_t) blockSize * xSzm[log2Width];
  int64_t numer = (int64_t) mWeight * ( (int64_t) x1yzm * blockSize - (int64_t) xSum * ySum );
  int32_t b1 = (int32_t)( ( numer < 0 ? numer - ( denom >> 1 ) : numer + ( denom >> 1 ) ) / denom );
  b1 = b1 < -32768 ? -32768 : ( b1 > 32767 ? 32767 : b1 );
  numer = (int64_t) mWeight * ( (int64_t) x2yzm * blockSize - (int64_t) xSum * ySum );
  int32_t b2 = (int32_t)( ( numer < 0 ? numer - ( denom >> 1 ) : numer + ( denom >> 1 ) ) / denom );
  b2 = b2 > 32767 ? 32767 : ( b2 < -32768 ? -32768 : b2 );
  const int32_t b0 = ( mWeight * ySum - ( b1 + b2 ) * xSum + ( blockSize >> 1 ) ) >> ( log2Width << 1 );
  if( b0 == 0 && b1 == 0 && b2 == 0 ) return;
  for( int y = 0; y < h; y++ )
    for( int x = 0; x < w; x++ )
    {
      const int32_t p = ( b0 + b1 * x + b2 * y + 256 ) >> 9;
      const int32_t z = dst[y * ds + x] - p;
      dst[y * ds + x] = (Pel)( z < 0 ? 0 : ( z > maxPel ? maxPel : z ) );
    }
}

static float orc_fast_exp( float n, float d )
{
  float x = 1.0f + n / ( d * 1024 );
  x *= x; x *= x; x *= x; x *= x; x *= x; x *= x; x *= x; x *= x; x *= x; x *= x;
  return x;
}

/* corrected: numRefs compact w*h blocks back to back */
void orc_mctf_apply_block( const Pel* src, int ss, Pel* dst, int ds, int w, int h, int bitDepth, const Pel* corrected, int numRefs,
                           const int32_t* verror, const double* refStrengths, double weightScaling, double sigmaSq )
{
  const int maxv = ( 1 << bitDepth ) - 1;
  int vnoise[16]; float vsw[16], vww[16];
  int minError = 0x7fffffff;
  for( int i = 0; i < numRefs; i++ )
  {
    int64_t variance = 0, diffsum = 0;
    const Pel* ref = corrected + (size_t) i * w * h;
    for( int y = 0; y < h; y++ )
      for( int x = 0; x < w; x++ )
      {
        const int diff = src[y * ss + x] - ref[y * w + x];
        variance += diff * diff;
        if( x != w - 1 ) { const int dR = src[y * ss + x + 1] - ref[y * w + x + 1]; diffsum += ( dR - diff ) * ( dR - diff ); }
        if( y != h - 1 ) { const int dD = src[( y + 1 ) * ss + x] - ref[( y + 1 ) * w + x]; diffsum += ( dD - diff ) * ( dD - diff ); }
      }
    variance *= (int64_t) 1 << ( 2 * ( 10 - bitDepth ) );
    diffsum  *= (int64_t) 1 << ( 2 * ( 10 - bitDepth ) );
    const int cntV = w * h, cntD = 2 * cntV - w - h;
    vnoise[i] = (int) round( ( 15.0 * cntD / cntV * variance + 5.0 ) / ( diffsum + 5.0 ) );
    if( verror[i] < minError ) minError = verror[i];
  }
  for( int i = 0; i < numRefs; i++ )
  {
    const int error = verror[i], noise = vnoise[i];
    float ww = 1, sw = 1;
    ww *= ( noise < 25 ) ? 1.0 : 0.6;
    sw *= ( noise < 25 ) ? 1.0 : 0.8;
    ww *= ( error < 50 ) ? 1.2 : ( ( error > 100 ) ? 0.6 : 1.0 );
    sw *= ( error < 50 ) ? 1.0 : 0.8;
    ww *= ( ( minError + 1.0 ) / ( error + 1.0 ) );
    vww[i] = ww * weightScaling * refStrengths[i];
    vsw[i] = sw * 2 * sigmaSq;
  }
  for( int y = 0; y < h; y++ )
    for( int x = 0; x < w; x++ )
    {
      const Pel orgVal = src[y * ss + x];
      float temporalWeightSum = 1.0;
      float newVal = (float) orgVal;
      for( int i = 0; i < numRefs; i++ )
      {
        const int refVal = corrected[(size_t) i * w * h + y * w + x];
        const int diff = refVal - orgVal;
        const float diffSq = diff * diff;
        float weight = vww[i] * orc_fast_exp( -diffSq, vsw[i] );
        newVal += weight * refVal;
        temporalWeightSum += weight;
      }
      newVal /= temporalWeightSum;
      Pel sampleVal = (Pel)( newVal + 0.5 );
      sampleVal = sampleVal < 0 ? 0 : ( sampleVal > maxv ? maxv : sampleVal );
      dst[y * ds + x] = sampleVal;
    }
}

double orc_mctf_calc_var( const Pel* org, int so, int w, int h )
{
  int avg = 0;
  for( int y = 0; y < h; y++ ) for( int x = 0; x < w; x++ ) avg += org[y * so + x];
  avg <<= 4;
  avg = avg / ( w * h );
  int64_t variance = 0;
  for( int y = 0; y < h; y++ ) for( int x = 0; x < w; x++ ) { const int pix = org[y * so + x] << 4; variance += ( pix - avg ) * ( pix - avg ); }
  return variance / 256.0;
}

/* Body of MCTF::xFinalizeBlkLine for one luma block (MCTF.cpp:1437-1483): per reference applyFrac (+ planar correction), then applyBlock.
 * refs[i]: pointer to sample (0,0) of reference picture i (same stride rs); mv[i] = { x, y, error, rmsme } in 1/16 pel. */
void orc_mctf_finalize_block( const Pel* orgPlane, int so, const Pel* const* refs, int rs, int numRefs, const int32_t* mv4, int bx, int by, int w, int h,
                              int bitDepth, int tap4, int planarEnabled, const double* refStrengths, double weightScaling, double sigmaSq, Pel* dstPlane, int ds )
{
  Pel* corrected = (Pel*) malloc( sizeof( Pel ) * numRefs * w * h );
  int32_t verror[16];
  for( int i = 0; i < numRefs; i++ )
  {
    const int32_t* mv = mv4 + 4 * i;
    const Pel* src = refs[i] + (ptrdiff_t)( by + ( mv[1] >> 4 ) ) * rs + bx + ( mv[0] >> 4 );
    Pel* dst = corrected + (size_t) i * w * h;
    orc_mctf_apply_frac( tap4, src, rs, dst, w, w, h, mv[0] & 15, mv[1] & 15, bitDepth );
    if( mv[3] > 0 && planarEnabled && w == h && w <= 32 )
      orc_mctf_planar_correction( orgPlane + (ptrdiff_t) by * so + bx, so, dst, w, w, h, bitDepth, (unsigned) mv[3] );
    verror[i] = mv[2];
  }
  orc_mctf_apply_block( orgPlane + (ptrdiff_t) by * so + bx, so, dstPlane + (ptrdiff_t) by * ds + bx, ds, w, h, bitDepth, corrected, numRefs, verror, refStrengths, weightScaling, sigmaSq );
  free( corrected );
}

/* ------------------------------------------------------------------------------------------------------
 * Fractional-pel refinement feeding SATD (SURVEY 8f rank 2): the filtered blocks InterSearch::xPatternRefinement evaluates
 * (EncoderLib/InterSearch.cpp:760-972; xExtDIFUpSamplingH/Q :2912,2973) are always produced by TWO passes of the 8-tap luma filter:
 * InterpolationFilter::filterHor(frac_x, isLast = false) then filterVer(frac_y, isFirst = false, isLast = true)
 * (CommonLib/InterpolationFilter.cpp:357-455 filter<N,...>, :258-340 filterCopy for frac 0, which equals the filter with the
 * tap 64).  Quarter-pel phases; the filter set follows m_meReduceTap (0: 8-tap m_lumaFilter, 1: 6-tap m_lumaFilter4x4, 2: 4-tap m_chromaFilter[frac<<1],
 * InterpolationFilter.cpp:557-600) and useAltHpelIf replaces the half-pel phase by m_lumaAltHpelIFilter.
 * ---------------------------------------------------------------------------------------------------- */
/* quarter-pel phases as 8-tap rows over pels x-3 .. x+4: [reduceTap][phase][tap]
 *   0: m_lumaFilter rows 0,4,8,12 (8 taps)   1: m_lumaFilter4x4 rows 4,8,12 used as 6 taps (:64-83, filter<6> skips entry 0)
 *   2: m_chromaFilter rows 8,16,24 (4 taps over x-1 .. x+2, :107-142; what every preset's ReduceFilterME = 2 selects)
 * alt: m_lumaAltHpelIFilter as 6 taps (:106), replaces the half-pel phase when useAltHpelIf */
static const int8_t luma_qpel_sets[3][4][8] = {
  { { 0, 0, 0, 64, 0, 0, 0, 0 }, { -1, 4, -10, 58, 17, -5, 1, 0 }, { -1, 4, -11, 40, 40, -11, 4, -1 }, { 0, 1, -5, 17, 58, -10, 4, -1 } },
  { { 0, 0, 0, 64, 0, 0, 0, 0 }, {  0, 3, -10, 58, 17, -5, 1, 0 }, {  0, 3, -11, 40, 40, -11, 3,  0 }, { 0, 1, -5, 17, 58, -10, 3,  0 } },
  { { 0, 0, 0, 64, 0, 0, 0, 0 }, {  0, 0,  -4, 54, 16, -2, 0, 0 }, {  0, 0,  -4, 36, 36,  -4, 0,  0 }, { 0, 0, -2, 16, 54,  -4, 0,  0 } } };
static const int8_t luma_alt_hpel[8] = { 0, 3, 9, 20, 20, 9, 3, 0 };
static const int8_t* qpel_taps( int reduceTap, int altHpel, int phase ) { return ( altHpel && phase == 2 ) ? luma_alt_hpel : luma_qpel_sets[reduceTap][phase]; }

/* src points at the integer position of the block; fx, fy in quarter pels (0..3) */
void orc_if_two_pass( const Pel* src, int ss, int w, int h, int fx, int fy, int bitDepth, int reduceTap, int altHpel, Pel* dst, int ds )
{
  const int8_t* cx = qpel_taps( reduceTap, altHpel, fx );
  const int8_t* cy = qpel_taps( reduceTap, altHpel, fy );
  const int headRoom = 14 - bitDepth > 2 ? 14 - bitDepth : 2;
  const int shift1 = 6 - headRoom, offset1 = -( 8192 << shift1 );
  const int shift2 = 6 + headRoom, offset2 = ( 1 << ( shift2 - 1 ) ) + ( 8192 << 6 );
  const int maxv = ( 1 << bitDepth ) - 1;
  int16_t* tmp = (int16_t*) malloc( sizeof( int16_t ) * ( h + 7 ) * w );
  for( int r = 0; r < h + 7; r++ )
    for( int x = 0; x < w; x++ )
    {
      const Pel* p = src + ( r - 3 ) * ss + x - 3;
      int sum = 0;
      for( int t = 0; t < 8; t++ ) sum += cx[t] * p[t];
      tmp[r * w + x] = (int16_t)( ( sum + offset1 ) >> shift1 );
    }
  for( int y = 0; y < h; y++ )
    for( int x = 0; x < w; x++ )
    {
      int sum = 0;
      for( int t = 0; t < 8; t++ ) sum += cy[t] * tmp[( y + t ) * w + x];
      const int v = ( sum + offset2 ) >> shift2;
      dst[y * ds + x] = (Pel)( v < 0 ? 0 : ( v > maxv ? maxv : v ) );
    }
  free( tmp );
}

/* Distortion table of all quarter-pel offsets (i, j) in -3..3 around the integer vector: out[b][j+3][i+3].
 * blk[b] = { x, y, w, h, mvx, mvy } (integer pel vector); family 1 = SAD, 2 = HAD (xGetHADs). */
void orc_frac_cost_grid( const Pel* orgPlane, int so, const Pel* refPlane, int sr, const int32_t* blk, int n, int family, int bitDepth, int reduceTap, int altHpel, uint32_t* out )
{
  Pel* pred = (Pel*) malloc( sizeof( Pel ) * 64 * 64 );
  for( int b = 0; b < n; b++ )
  {
    const int32_t* d = blk + 6 * (size_t) b;
    const int w = d[2], h = d[3];
    const Pel* org = orgPlane + (ptrdiff_t) d[1] * so + d[0];
    for( int j = -3; j <= 3; j++ )
      for( int i = -3; i <= 3; i++ )
      {
        const Pel* src = refPlane + (ptrdiff_t)( d[1] + d[5] + ( j >> 2 ) ) * sr + d[0] + d[4] + ( i >> 2 );
        orc_if_two_pass( src, sr, w, h, i & 3, j & 3, bitDepth, reduceTap, altHpel, pred, w );
        out[( (size_t) b * 7 + ( j + 3 ) ) * 7 + ( i + 3 )] = (uint32_t) orc_dist( family, org, so, pred, w, w, h, 0 );
      }
  }
  free( pred );
}

/* ------------------------------------------------------------------------------------------------------
 * Affine gradient helpers (CommonLib/AffineGradientSearch.cpp:84-190)
 * ---------------------------------------------------------------------------------------------------- */
void orc_sobel( int vertical, const Pel* p, int ps, Pel* d, int ds, int w, int h )
{
  for( int j = 1; j < h - 1; j++ )
    for( int k = 1; k < w - 1; k++ )
    {
      const Pel* c = p + j * ps + k;
      int v;
      if( !vertical ) v = c[1 - ps] - c[-1 - ps] + ( c[1] << 1 ) - ( c[-1] << 1 ) + c[1 + ps] - c[-1 + ps];
      else            v = c[ps - 1] - c[-ps - 1] + ( c[ps] << 1 ) - ( c[-ps] << 1 ) + c[ps + 1] - c[-ps + 1];
      d[j * ds + k] = (Pel) v;
    }
  /* border replication: edges copy their inner neighbour, corners copy the inner diagonal (:101-114) */
  for( int j = 1; j < h - 1; j++ ) { d[j * ds] = d[j * ds + 1]; d[j * ds + w - 1] = d[j * ds + w - 2]; }
  for( int k = 1; k < w - 1; k++ ) { d[k] = d[ds + k]; d[( h - 1 ) * ds + k] = d[( h - 2 ) * ds + k]; }
  d[0] = d[ds + 1]; d[w - 1] = d[ds + w - 2];
  d[( h - 1 ) * ds] = d[( h - 2 ) * ds + 1]; d[( h - 1 ) * ds + w - 1] = d[( h - 2 ) * ds + w - 2];
}

void orc_equal_coeff( int sixParam, const Pel* resi, int rs, const Pel* gx, const Pel* gy, int ds, int w, int h, int64_t* eq )
{
  const int np = sixParam ? 6 : 4;
  for( int j = 0; j < h; j++ )
  {
    const int cy = ( ( j >> 2 ) << 2 ) + 2;
    for( int k = 0; k < w; k++ )
    {
      const int cx = ( ( k >> 2 ) << 2 ) + 2;
      const int a = gx[j * ds + k], b = gy[j * ds + k];
      int c[6];
      if( !sixParam ) { c[0] = a; c[1] = cx * a + cy * b; c[2] = b; c[3] = cy * a - cx * b; }
      else            { c[0] = a; c[1] = cx * a; c[2] = b; c[3] = cx * b; c[4] = cy * a; c[5] = cy * b; }
      for( int col = 0; col < np; col++ )
      {
        for( int row = 0; row < np; row++ ) eq[( col + 1 ) * 7 + row] += (int64_t) c[col] * c[row];
        eq[( col + 1 ) * 7 + np] += ( (int64_t) c[col] * resi[j * rs + k] ) * 8;
      }
    }
  }
}
