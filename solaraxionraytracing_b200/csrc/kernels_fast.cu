// kernels_fast.cu — the "fast" fused Monte Carlo kernel (precision mode 1), sm_100a.
//
// Same physics as traceAxion (src/raytracer.nim:1736-2221) but formulated for throughput instead of for bitwise
// agreement with the reference's operation order:
//   * the ray is carried as (point on the exit disc of the magnetic field, slopes dx/dz, dy/dz) instead of two
//     points 1.5e14 mm apart, which removes the catastrophic cancellation the reference suffers at solar
//     distances (DESIGN.md "Numerical floor") — geometry is FP64 *algebra* only: no FP64 transcendental, and every
//     FP64 divide / sqrt is an FP32 MUFU seed plus one Newton step in FP64 (relative error ~1e-14);
//   * the reflection is written without trigonometry: with s = n.v (unit normal, unit ray) the reference's
//     "rotate v by 2*alpha about n x v" (rt:762-780) is v' = v (1 - 2 s^2 + 2 |s| s) - 2 |s| n;
//   * everything that only scales the weight (emission direction sines, grazing angles for the reflectivity
//     lookup, cos(yaw), transmissions) is FP32 with MUFU intrinsics; transmissions, the energy and the reflectivity
//     cell of each of the nE tabulated energies come from a per-energy-index LUT built once at sart_create;
//   * the two inverse-CDF searches (rt:437, 464) are exact integer work: cdf[i] < u with u = (w + 0.5) 2^-32 is
//     w >= T[i] for the 32-bit threshold T[i] = smallest such w, so the f64 tables become u32 tables of half the size,
//     a guide table (bucket = top bits of w) gives the start, one or two 16-byte loads give 8 thresholds and the index
//     is start + the number of thresholds <= w — no loop, no f64 compare, same index as lowerBound on the f64 CDF;
//     the dependent loads are issued ahead of the geometry that separates them from their use;
//   * run-wide tables (radius CDF, guide, shell constants) are staged once per block in shared memory;
//   * counters live in registers / per-warp shared memory and are flushed once per block.
// Exit codes follow the same decision sequence as the exact pipeline, so the counters of both are comparable.
#include "fast_common.cuh"

namespace sart {
namespace fast {

// The two fused kernels run one block of kBlockF threads per SM (24 warps, 76-78 registers: the register file allows no
// more), so that the per-block tables exist once per SM and the shared memory saved goes to L1 (see kernels_f32.cu);
// the per-ray and mass-scan kernels keep kBlock = 256.
#ifndef SART_FAST_BLOCK_FUSED
#define SART_FAST_BLOCK_FUSED 768
#endif
constexpr int kBlockF = SART_FAST_BLOCK_FUSED, kWarpsF = kBlockF / 32;

// Root choice of findPos* (rt:646-658): roots of A t^2 + 2 hb t + C = 0 in the reference's order root1 = (-hb - sq)/A,
// root2 = (-hb + sq)/A, each accepted only if zmin < pz + t dz < zmax. With q = -(hb + sign(hb) sq) the roots are q/A
// (the larger in magnitude) and C/q. The large root is never inside a mirror in practice (it is metres away), so it is
// excluded with a division-free bound and only then does the small root need a reciprocal; the rare other case
// reproduces the reference's order exactly.
static __device__ __noinline__ bool pick_root_slow(double A, double q, double C, bool first_is_qA, double dz, double lo,
                                            double hi, double& t) {
  auto in_range = [&](double num, double den) {
    const double nd = num * dz;  // lo < (num/den) dz < hi without dividing
    return den > 0.0 ? (nd > lo * den && nd < hi * den) : (nd < lo * den && nd > hi * den);
  };
  const bool okA = in_range(q, A), okC = in_range(C, q);
  double num, den;
  if (first_is_qA ? okA : okC) { num = first_is_qA ? q : C; den = first_is_qA ? A : q; }
  else if (first_is_qA ? okC : okA) { num = first_is_qA ? C : q; den = first_is_qA ? q : A; }
  else return false;
  t = num / den;
  return true;
}
__device__ __forceinline__ bool pick_root(double A, double hb, double C, double pz, double dz, double zmin, double zmax,
                                          double& t) {
  const double disc = fma(hb, hb, -A * C);
  if (!(disc >= 0.0)) return false;
  const double sq = disc > 1e-30 ? disc * rsqrt_nr(disc) : 0.0;
  const double q = -(hb + copysign(sq, hb));
  const double lo = zmin - pz, hi = zmax - pz;
  if (fabs(q * dz) < fmax(fabs(lo), fabs(hi)) * fabs(A)) return pick_root_slow(A, q, C, hb >= 0.0, dz, lo, hi, t);
  const double ts = C * rcp_nr(q);
  const double zs = ts * dz;
  t = ts;
  return zs > lo && zs < hi;
}

// Reflection of unit vector v off unit normal n (rt:762-780 without trigonometry); returns |n.v| = sin(alpha).
__device__ __forceinline__ double reflect(D3 n, D3& v) {
  const double s = n.x * v.x + n.y * v.y + n.z * v.z;
  const double as = fabs(s);
  const double f = fma(2.0 * as, s, fma(-2.0 * s, s, 1.0));  // 1 - 2 s^2 + 2 |s| s
  v.x = fma(v.x, f, -2.0 * as * n.x);
  v.y = fma(v.y, f, -2.0 * as * n.y);
  v.z = fma(v.z, f, -2.0 * as * n.z);
  return as;
}

// Shared-memory tables of one block (shells first so their addresses are compile-time offsets).
struct Smem {
  const ShellFast* shell;
  const uint32_t* radThr;     // [thrPitch(nRadii)] thresholds of the radius CDF, 16-byte aligned
  const uint16_t* radGuide;   // [kRadGuide]
  const uint8_t* shellGuide;
};
__host__ __device__ __forceinline__ size_t align16(size_t n) { return (n + 15) & ~size_t(15); }
__device__ __forceinline__ size_t smem_layout(const FastParams& P, unsigned char* base, Smem& s, unsigned char*& tail) {
  size_t off = 0;
  s.shell = reinterpret_cast<const ShellFast*>(base + off); off += align16(size_t(P.nShells) * sizeof(ShellFast));
  s.radThr = reinterpret_cast<const uint32_t*>(base + off); off += size_t(thr_pitch(P.nRadii)) * 4;
  s.radGuide = reinterpret_cast<const uint16_t*>(base + off); off += size_t(kRadGuide) * 2;
  s.shellGuide = base + off; off += align16(size_t(P.nShellGuide));
  tail = base + off;
  return off;
}
__device__ __forceinline__ void smem_fill(const FastParams& P, const FastTables& T, const Smem& s) {
  for (int i = threadIdx.x; i < P.nShells * int(sizeof(ShellFast) / 8); i += blockDim.x)
    reinterpret_cast<double*>(const_cast<ShellFast*>(s.shell))[i] = reinterpret_cast<const double*>(T.shells)[i];
  if (P.nRadii > 0) {
    for (int i = threadIdx.x; i < thr_pitch(P.nRadii); i += blockDim.x) const_cast<uint32_t*>(s.radThr)[i] = T.radiusThr[i];
    for (int i = threadIdx.x; i < kRadGuide / 8; i += blockDim.x)   // 16 bytes per thread and step
      reinterpret_cast<uint4*>(const_cast<uint16_t*>(s.radGuide))[i] = __ldg(reinterpret_cast<const uint4*>(T.radiusGuide) + i);
  }
  for (int i = threadIdx.x; i < P.nShellGuide; i += blockDim.x) const_cast<uint8_t*>(s.shellGuide)[i] = T.shellGuide[i];
}

// A ray that survived everything before the mirrors (stage A): what stage B needs to finish it. 48 bytes; this is
// the record the compacting kernel queues in shared memory.
struct Rec {
  double x0, y0, tx, ty;   // pointEntranceXRT (telescope frame, z = 0) and slopes dx/dz, dy/dz
  double path2;            // pathCB^2
  int hitLayer, eIdx;
  bool clamped;
};

// Stage A of traceAxion: sampling, bore/pipe clipping, telescope frame, opaque structures, shell (rt:1754-1957).
// Returns the exit code of an early return, or -1 with `rec` filled.
template <bool kWolter>
__device__ __forceinline__ int stage_a(const FastParams& P, const FastTables& T, const Smem& S, uint64_t seed,
                                       uint64_t ray, Rec& rec) {
  const ShellFast* __restrict__ sShell = S.shell;
  uint32_t w[6];
  ray_words(seed, ray, w);
  constexpr float k2m32 = 2.3283064365386963e-10f;  // 2^-32
  bool clamped = false;

  // ================= sampling rt:1754-1764 (or the X-ray test source rt:1765-1801)
  double ex, ey, sx, sy;   // point on the exit disc of the field (z = lengthB) and slopes
  int eIdx;
  // energy search state: the guide entry is loaded here, the thresholds after the clip tests and the index is resolved
  // at the end of the stage — the dependent global loads overlap the geometry instead of stalling in a row
  int e0 = 0;
  const uint32_t* eRow = nullptr;
  if (!P.testXray) {
    // emission shell rt:437: rIdx = lowerBound(fluxRadiusCDF, u), exact (integer thresholds in shared memory)
    int rIdx;
    {
      const uint32_t wr = w[2];
      const int r0 = int(S.radGuide[wr >> (32 - kRadGuideBits)]) & ~3;
      rIdx = r0 + count_le(*reinterpret_cast<const uint4*>(S.radThr + r0), wr);
      if (rIdx == r0 + 4) {
        rIdx += count_le(*reinterpret_cast<const uint4*>(S.radThr + r0 + 4), wr);
        if (rIdx == r0 + 8) rIdx = thr_search_tail(S.radThr, r0 + 8, P.nRadii, wr);
      }
      if (wr == 0xffffffffu) rIdx = lower_bound_window(T.radiusCDF, 0, P.nRadii, u01(wr));   // saturated thresholds
      if (rIdx > P.nRadii - 1) rIdx = P.nRadii - 1;
    }
    {
      const uint32_t we = w[5];
      e0 = int(__ldg(T.energyGuide + size_t(rIdx) * kEnGuide + (we >> (32 - kEnGuideBits)))) & ~3;
      eRow = T.energyThr + size_t(rIdx) * thr_pitch(P.nEnergies);
    }
    const float rs = (0.0015f + float(rIdx) * 0.0005f);  // fraction of the solar radius (weight-free: direction only)
    float s1, c1, s2, c2;
    sincos_2pi(float(w[0]) * k2m32, s1, c1);              // phi = 360 u0
    __sincosf(3.14159265358979f * (float(w[1]) * k2m32), &s2, &c2);  // theta = 180 u1 (uniform in theta, quirk Q7)
    const double rsun = double(rs) * P.radiusSun;
    const double Ox = rsun * double(c1 * s2), Oy = rsun * double(s1 * s2), Ozr = rsun * double(c2);
    // exit disc rt:412-422
    float sd, cd;
    sincos_2pi(float(w[4]) * k2m32, sd, cd);
    const float rd = sqrtf((float(w[3]) + 0.5f) * k2m32);
    ex = P.radiusCB * double(rd * cd);
    ey = P.radiusCB * double(rd * sd);
    const double invD = rcp_nr(P.lengthB + P.sunDist - Ozr);  // lengthB - O.z
    sx = (ex - Ox) * invD;
    sy = (ey - Oy) * invD;
    // (energy: the reference recovers the radius index from the emission point, rt:454-460; it is rIdx again)
    eIdx = 0;
  } else {
    float sd, cd;
    sincos_2pi(float(w[1]) * k2m32, sd, cd);
    const float rd = sqrtf((float(w[0]) + 0.5f) * k2m32);
    const double Ox = P.srcX + P.srcRadius * double(rd * cd), Oy = P.srcY + P.srcRadius * double(rd * sd);
    if (P.parallelSource) {
      ex = Ox + (0.5 * u01(w[2]) - 0.25);
      ey = Oy + (0.5 * u01(w[3]) - 0.25);
    } else {
      sincos_2pi(float(w[3]) * k2m32, sd, cd);
      const float r2 = sqrtf((float(w[2]) + 0.5f) * k2m32);
      ex = P.radiusCB * double(r2 * cd);
      ey = P.radiusCB * double(r2 * sd);
    }
    const double invD = rcp_nr(P.lengthB - P.srcZ);
    sx = (ex - Ox) * invD;
    sy = (ey - Oy) * invD;
    // collimator rt:1800: point at z = colZ relative to the source centre
    const double qx = fma(sx, P.colDz, Ox) - P.srcX, qy = fma(sy, P.colDz, Oy) - P.srcY;
    eIdx = P.srcEIdx;
    if (!(qx * qx + qy * qy < P.srcRadius2)) return SART_EXIT_COLLIMATOR;
  }

  // ================= bore and pipes rt:1813-1872: points of the line at the clip planes
  const double s2sum = fma(sx, sx, sy * sy);
  const double p0x = fma(-sx, P.lengthB, ex), p0y = fma(-sy, P.lengthB, ey);
  const bool hitEntrance = fma(p0x, p0x, p0y * p0y) < P.radiusCB2;
  const double pex = fma(sx, P.dzExitCB, ex), pey = fma(sy, P.dzExitCB, ey);
  const bool insideExit = fma(pex, pex, pey * pey) < P.radiusCB2;
  if (!insideExit) return hitEntrance ? SART_EXIT_CLIP_EXIT_CB : SART_EXIT_MISSED_BORE;
  // (a ray that misses the entrance disc but is inside at the exit entered through the wall exactly once)
  double path2;  // pathCB^2 rt:1843
  if (hitEntrance) {
    path2 = P.lengthB * P.lengthB * (1.0 + s2sum);
  } else {
    // wall crossing |e + s t|^2 = R^2, t < 0
    const double hb = fma(ex, sx, ey * sy), c = fma(ex, ex, ey * ey) - P.radiusCB2;
    const double disc = fma(hb, hb, -s2sum * c);
    const double sq = disc > 1e-30 ? disc * rsqrt_nr(disc) : 0.0;
    const double t1 = (hb >= 0.0) ? -(hb + sq) * rcp_nr(s2sum) : c * rcp_nr(sq - hb);
    path2 = t1 * t1 * (1.0 + s2sum);
  }
  {
    const double qx = fma(sx, P.dzPipe1, ex), qy = fma(sy, P.dzPipe1, ey);
    if (!(fma(qx, qx, qy * qy) < P.rPipe12)) return SART_EXIT_CLIP_PIPE_VT3;
  }
  double x0 = fma(sx, P.dzPipe2, ex), y0 = fma(sy, P.dzPipe2, ey);
  if (!(fma(x0, x0, y0 * y0) < P.rPipe12)) return SART_EXIT_CLIP_PIPE_XRT;  // quirk Q2
  // energy thresholds: 8 entries from the 16-byte aligned entry at or below the guide's start (windows are 1-2 wide)
  uint4 etA = make_uint4(0, 0, 0, 0);
  if (eRow) etA = __ldg(reinterpret_cast<const uint4*>(eRow + e0));

  // ================= telescope frame rt:1888-1905 (rotation about (0, 0, halfLenTel); identity when not turned)
  double dx = sx, dy = sy, dz = 1.0, z0 = 0.0;
  if (P.rotated) {
    // rotateInX then rotateInY of point (x0, y0, 0) and of the direction
    double zt = 0.0 - P.halfLenTel;
    double xr = x0 * P.cosTX + zt * P.sinTX, zr = zt * P.cosTX - x0 * P.sinTX;
    double yr = y0 * P.cosTY - zr * P.sinTY;
    zr = zr * P.cosTY + y0 * P.sinTY;
    x0 = xr; y0 = yr; z0 = zr + P.halfLenTel;
    double ddx = dx * P.cosTX + dz * P.sinTX, ddz = dz * P.cosTX - dx * P.sinTX;
    double ddy = dy * P.cosTY - ddz * P.sinTY;
    ddz = ddz * P.cosTY + dy * P.sinTY;
    dx = ddx; dy = ddy; dz = ddz;
  }
  x0 -= P.oeX; y0 -= P.oeY;
  // renormalise to dz = 1 and move to the plane z = 0
  const double invdz = (dz == 1.0) ? 1.0 : rcp_nr(dz);
  const double tx = dx * invdz, ty = dy * invdz;  // slopes in the telescope frame
  x0 = fma(-z0, tx, x0); y0 = fma(-z0, ty, y0);   // pointEntranceXRT
  const double rho0sq = fma(x0, x0, y0 * y0);
  const double invRho0 = rsqrt_nr(rho0sq);
  const double radialDist = rho0sq * invRho0;

  // ================= opaque structures rt:1635-1704
  if (kWolter) {
    const bool xmm = P.telKind == SART_TK_XMM;
    bool hit = false;
    const float zs = xmm ? -85.0f : -35.0f;
    const float phiF = acosf(float(x0 * invRho0)) * 57.29577951308232f;
    const float xs = float(fma(double(zs), tx, x0)), ys = float(fma(double(zs), ty, y0));
    const float phiS = acosf(xs * rsqrtf(xs * xs + ys * ys)) * 57.29577951308232f;
    if (xmm) {
      if (radialDist <= 64.7) {
        hit = true;   // htNone: the centre is opaque; other hole types open a pattern of holes in it (rt:1674-1688)
        if (P.holeType != SART_HT_NONE) {
          double edge;
          hit = !in_hole(P.holeType, P.numberOfHoles, P.holeInOptics, x0, y0, edge);
        }
      }
      else if (radialDist < 151.6 && radialDist > (151.6 - 20.9)) hit = true;
      else {
        // |phi - 22.5 k| <= 1.145 for some k in 0..16 (phi in [0, 180])
        const float a = fabsf(phiF - 22.5f * rintf(phiF * (1.0f / 22.5f)));
        const float b = fabsf(phiS - 22.5f * rintf(phiS * (1.0f / 22.5f)));
        hit = (a <= 1.145f) || (b <= 1.145f);
      }
    } else {
      if (radialDist < 37.5) hit = true;
      else {
        const float a = fabsf(phiF - 60.0f * rintf(phiF * (1.0f / 60.0f)));
        const float b = fabsf(phiS - 60.0f * rintf(phiS * (1.0f / 60.0f)));
        hit = (a <= 3.75f) || (b <= 3.75f);
      }
    }
    if (hit) return SART_EXIT_OPAQUE;
  }

  // ================= shell rt:1932-1957: uniform radial guide + at most one forward step
  const int nS = P.nShells;
  if (radialDist > sShell[nS - 1].R1) return SART_EXIT_OUTSIDE_SHELLS;
  int hitLayer;
  {
    int b = int((radialDist - P.shellRhoMin) * P.shellInvStep);
    b = b < 0 ? 0 : (b > P.nShellGuide - 1 ? P.nShellGuide - 1 : b);
    hitLayer = S.shellGuide[b];
    while (hitLayer < nS - 1 && !(sShell[hitLayer].R1 > radialDist)) ++hitLayer;   // first j with R1[j] > radialDist
    if (!(sShell[hitLayer].R1 > radialDist)) return SART_EXIT_NO_MIRROR_HIT;  // == R1[last]
    if (hitLayer > 0 && radialDist < sShell[hitLayer - 1].R1pT) {   // R1[j-1] < radialDist holds by construction
      if (radialDist > sShell[hitLayer - 1].R1) return SART_EXIT_GLASS_FRONT;
    }
  }
  // energy index rt:464 from the thresholds loaded above: idx = lowerBound(diffFluxCDFs[iRad], u), exact
  if (eRow) {
    const uint32_t we = w[5];
    eIdx = e0 + count_le(etA, we);
    if (eIdx == e0 + 4) {   // ~1 ray in 8: the next four thresholds, loaded only by the lanes that need them (one divergent
                            // gather less per ray than loading them with etA: CAST+LLNL 35.2 -> 32.8 ms)
      eIdx += count_le(__ldg(reinterpret_cast<const uint4*>(eRow + e0 + 4)), we);
      if (eIdx == e0 + 8) eIdx = thr_search_tail(eRow, e0 + 8, P.nEnergies, we);
    }
    if (we == 0xffffffffu)   // saturated thresholds: the f64 row decides
      eIdx = lower_bound_window(T.energyCDF + size_t(eRow - T.energyThr) / thr_pitch(P.nEnergies) * P.nEnergies, 0, P.nEnergies, u01(we));
    if (eIdx > P.nEnergies - 1) { eIdx = P.nEnergies - 1; clamped = true; }
  }
  rec.x0 = x0; rec.y0 = y0; rec.tx = tx; rec.ty = ty; rec.path2 = path2;
  rec.hitLayer = hitLayer; rec.eIdx = eIdx; rec.clamped = clamped;
  return -1;
}

// Stage B: the two reflections, nickel / degenerate exits, detector plane, weights, window (rt:1971-2221).
// The outcome goes to `sink` at the point where it is known — sink.fail(code) for a geometric exit, sink.hit(record)
// for a ray that reached the weight stage — instead of through a result struct merged over all return paths (that
// merge cost ~10 % of the kernel's instructions in register moves and zero fills).
// Sink::kFold: fold the conversion probability of the single axion mass sink.m2 into wPre right away.
template <bool kWolter, class Sink>
__device__ __forceinline__ void stage_b(const FastParams& P, const FastTables& T, const Smem& S, const Rec& rec,
                                        Sink& sink) {
  const ShellFast* __restrict__ sShell = S.shell;
  RayResult out;
  out.convVac = 1.f; out.gasGamma = 0.f; out.gasE1 = 0.f; out.gasE2 = 0.f; out.gasInv2E = 0.f; out.gasL = 0.0;
  const double x0 = rec.x0, y0 = rec.y0, tx = rec.tx, ty = rec.ty, path2 = rec.path2;
  const int hitLayer = rec.hitLayer, eIdx = rec.eIdx;
  bool clamped = rec.clamped;
  const float4 elv = __ldg(reinterpret_cast<const float4*>(T.elut) + eIdx);   // needed at the weight stage
  const EnergyLUT el = {__float_as_int(elv.x), elv.y, elv.z, elv.w};
  const double rho0sq = fma(x0, x0, y0 * y0);
  const double t2sum = fma(tx, tx, ty * ty);
  const double invLen = rsqrt_nr(1.0 + t2sum);
  const ShellFast& sh = sShell[hitLayer];
  const double lM = P.lMirror;
  const double below = hitLayer > 0 ? sShell[hitLayer - 1].R1pT : 0.0;

  // ================= mirror 1 rt:1983-2020. Ray: (x0 + tx z, y0 + ty z, z).
  double z1;
  bool hit1;
  if (kWolter) {   // paraboloid rho^2 = r3^2 + e (l - z)  (findPosParabolic rt:660-690)
    hit1 = pick_root(t2sum, fma(x0, tx, y0 * ty) + 0.5 * sh.p_e, rho0sq - sh.p_c0, 0.0, 1.0, 0.0, sh.zmax1, z1);
  } else {         // cone rho = r1 - tan(beta) z  (findPosCone rt:628-658)
    hit1 = pick_root(t2sum - sh.tan1 * sh.tan1, fma(x0, tx, y0 * ty) + sh.tan1 * sh.R1, rho0sq - sh.r1sq, 0.0, 1.0,
                     0.0, sh.zmax1, z1);
  }
  if (!hit1) {
    // The reference carries on with pointMirror1 = pointExitCB (start point returned, rt:655-658) and reaches the
    // nickel test before the degenerate-hit test (rt:2040-2057): reproduce which of the two exits it takes.
    int code = SART_EXIT_NO_MIRROR_HIT;
    if (hitLayer > 0) {
      double zc = P.zExitCBtel;  // pointExitCB.z in the telescope frame
      if (P.rotated) {   // turned: the z of the ray's point whose laboratory z is zExitCB (trace_f32.cuh: exit_plane_z32)
        const double r13 = P.sinTX, r23 = -P.cosTX * P.sinTY, r33 = P.cosTX * P.cosTY, h = P.halfLenTel;
        zc = (fma(r33, h, P.zExitCBtel - h) - fma(r13, x0 + P.oeX, r23 * (y0 + P.oeY))) * rcp_nr(fma(r13, tx, fma(r23, ty, r33)));
      }
      const double xc = fma(zc, tx, x0), yc = fma(zc, ty, y0);
      const double rc2 = fma(xc, xc, yc * yc);
      const double rc = rc2 * rsqrt_nr(rc2);
      double nz;
      if (kWolter) nz = rc * sh.p_r3tan * rsqrt_nr(fmax(fma(sh.p_e, lM - zc, sh.p_r3sq), 1e-300));
      else nz = sh.tan1 * rc;
      const double sg = (fma(xc, tx, yc * ty) + nz) * invLen * rsqrt_nr(fma(rc, rc, nz * nz));
      const double a = fabs(sg);
      const double lhs = a * (lM - zc), rhs = sh.R1 - below;
      if (lhs * lhs > rhs * rhs * (1.0 - a * a)) code = SART_EXIT_NICKEL;
    }
    sink.fail(code);
    return;
  }
  D3 pm = {fma(tx, z1, x0), fma(ty, z1, y0), z1};
  D3 v = {tx * invLen, ty * invLen, invLen};
  double sinA1;
  {
    const double rr = fma(pm.x, pm.x, pm.y * pm.y);
    const double ir = rsqrt_nr(rr);
    D3 n;
    if (kWolter) {  // calcNormalVec msParabolic rt:740-746: n = (x, y, rho r3 tan / sqrt(r3^2 + e (l - z)))
      const double nz = sh.p_r3tan * rsqrt_nr(fma(sh.p_e, lM - pm.z, sh.p_r3sq));
      const double il = rsqrt_nr(1.0 + nz * nz);
      n = {pm.x * ir * il, pm.y * ir * il, nz * il};
    } else {        // msCone rt:737-739: n = (x, y, tan(beta) rho) / |.|
      n = {pm.x * ir * sh.cosb, pm.y * ir * sh.cosb, sh.sinb};
    }
    sinA1 = reflect(n, v);
  }
  // ================= mirror 2 rt:1994-2029. Ray: pm + t v.
  double t2;
  bool hit2;
  if (kWolter) {  // hyperboloid rho^2 = r3^2 + e (l - z) + g (l - z)^2  (findPosHyperbolic rt:692-729)
    const double u = lM - pm.z;
    const double A = fma(v.x, v.x, v.y * v.y) - sh.h_g * v.z * v.z;
    const double hb = fma(pm.x, v.x, pm.y * v.y) + (sh.h_g * u + 0.5 * sh.h_e) * v.z;
    const double C = fma(pm.x, pm.x, pm.y * pm.y) - sh.h_r3sq - (sh.h_e + sh.h_g * u) * u;
    hit2 = pick_root(A, hb, C, pm.z, v.z, sh.dm, sh.zmax2, t2);
  } else {        // cone rho = r4 - tan(3 beta) (z - distanceMirrors)
    const double rc = sh.r4 - sh.tan2 * (pm.z - sh.dm);
    const double A = fma(v.x, v.x, v.y * v.y) - sh.tan2 * sh.tan2 * v.z * v.z;
    const double hb = fma(pm.x, v.x, pm.y * v.y) + sh.tan2 * rc * v.z;
    const double C = fma(pm.x, pm.x, pm.y * pm.y) - rc * rc;
    hit2 = pick_root(A, hb, C, pm.z, v.z, sh.dm, sh.zmax2, t2);
  }
  // ================= nickel of the shell below rt:1706-1734: tan(alpha1) > (r1 - below)/(l - z1)
  if (hitLayer > 0) {
    // squared form of tan(alpha1) > (r1 - below)/(l - z1); both sides are positive
    const double lhs = sinA1 * (lM - z1), rhs = sh.R1 - below;
    if (lhs * lhs > rhs * rhs * (1.0 - sinA1 * sinA1)) { sink.fail(SART_EXIT_NICKEL); return; }
  }
  if (!hit2) { sink.fail(SART_EXIT_NO_MIRROR_HIT); return; }  // pointMirror2 == pointMirror1 (rt:2055)
  pm.x = fma(t2, v.x, pm.x); pm.y = fma(t2, v.y, pm.y); pm.z = fma(t2, v.z, pm.z);
  double sinA2;
  {
    const double rr = fma(pm.x, pm.x, pm.y * pm.y);
    const double ir = rsqrt_nr(rr);
    D3 n;
    if (kWolter) {  // msHyperbolic rt:747-758: n = (x, y, rho / m)
      const double u = lM - pm.z;
      const double q1 = 1.0 + 2.0 * u * sh.h_inv_nden, q2 = 1.0 + u * sh.h_inv_nden;
      const double nz = sh.h_r3tan * q1 * rsqrt_nr(fma(2.0 * sh.h_r3tan * u, q2, sh.h_r3sq));
      const double il = rsqrt_nr(1.0 + nz * nz);
      n = {pm.x * ir * il, pm.y * ir * il, nz * il};
    } else {
      n = {pm.x * ir * sh.cos3b, pm.y * ir * sh.cos3b, sh.sin3b};
    }
    sinA2 = reflect(n, v);
  }
  // ================= detector plane rt:797-814
  double xw, yw, zw;
  {
    const double ax = pm.x * P.cosPipe + pm.z * P.sinPipe - P.dShift, az = pm.z * P.cosPipe - pm.x * P.sinPipe;
    const double wx = v.x * P.cosPipe + v.z * P.sinPipe, wz = v.z * P.cosPipe - v.x * P.sinPipe;
    const double iwz = rcp_nr(wz);
    const double n = (sh.ddWin - az) * iwz;
    xw = fma(n, wx, ax); yw = fma(n, v.y, pm.y); zw = fma(n, wz, az);
    out.devDet = float(fabs(P.depthOverCos * iwz) * sqrt(fma(wx, wx, v.y * v.y)));   // deviationDet rt:2081-2085
  }
  xw -= P.lateralShift; yw -= P.transversalShift;
  // ================= weights rt:2101-2128 (mass-independent factors; P(a->gamma) is applied in finish_ray)
  out.eIdx = eIdx;
  {
    const float ya = -atan_small(float(ty)) * 57.29577951308232f;  // degrees; fed to cos as radians (quirk Q3)
    out.yaw = ya;
    float pre = __cosf(ya);
    const float path2f = float(path2);
    out.path = sqrtf(path2f);
    if (P.stage == SART_SK_VACUUM) {
      out.convVac = P.convK * path2f;              // conversionProb rt:363-365
    } else {
      const float2 gv = __ldg(reinterpret_cast<const float2*>(T.glut) + eIdx);
      const float pathm = sqrtf(path2f) * 1e-3f;
      const double gamma = P.gasGamma0 * double(gv.x);   // am:75-100
      out.gasL = double(pathm) / 1.97e-7;
      const float gl = float(gamma * out.gasL);
      out.gasGamma = float(gamma);
      out.gasE1 = -expm1f(-0.5f * gl); out.gasE2 = __expf(-0.5f * gl);   // 1 - e^(-Gamma L / 2) without cancellation, e^(-Gamma L / 2)
      out.gasInv2E = gv.y;
      const float distPipe = float(zw - P.zExitCBtel) * 1e-3f;   // intensitySuppression2 am:102-113
      pre *= __expf(-gv.x * float(P.gasRhoPipe100) * distPipe) * __expf(-gv.x * float(P.gasRhoMagnet100) * pathm);
    }
    out.pre = pre;
    double refl = 1.0;   // the product of two FP32 reflectivities can leave the FP32 range
    const float a1 = asin_small(float(sinA1)) * 57.29577951308232f, a2 = asin_small(float(sinA2)) * 57.29577951308232f;
    out.a1 = a1; out.a2 = a2;
    if (P.reflKind == SART_RK_EFFECTIVE_AREA) {
      if (!(P.flags & SART_CF_IGNORE_REFLECTION)) {   // rt:1553-1562; pitch = acos(-v.x) - 90 deg = asin(v.x) of the incoming ray
        const float sp = float(tx * invLen);
        const float pitch = (fabsf(sp) > 0.1f ? asinf(sp) : asin_small(sp)) * 57.29577951308232f;
        clamped |= (el.sbExp & (kLutClampRefl << 16)) != 0;   // the ray's energy lies outside the transmission table
        refl = double(__ldg(T.telTrans + eIdx)) * double(eff_area_angles(pitch, ya));
      }
    } else if (!(P.flags & SART_CF_IGNORE_REFLECTION)) {
      const float* zt = T.reflE + (size_t(sh.coat & kCoatMask) * (P.nEnergies + 1) + eIdx) * P.nAngles;
      clamped |= (sh.coat & kCoatClamped) != 0;
      clamped |= (el.sbExp & (kLutClampRefl << 16)) != 0;   // the ray's energy lies outside the reflectivity grid
      refl = double(refl_lookup(P, zt, a1, clamped)) * double(refl_lookup(P, zt, a2, clamped));
    }
    out.refl = refl;
    out.agas = el.Agas;
    out.wPre = refl * double(pre);   // FP32 factors, FP64 product: tiny weights must not flush to zero
    if (Sink::kFold) out.wPre *= conv_factor(P, out.convVac, out.gasGamma, out.gasE1, out.gasE2, out.gasInv2E, out.gasL, sink.m2);
  }
  out.clamped = clamped;
  out.shell = hitLayer;
  out.code = -1;
  // ================= window aperture rt:2139-2147
  const double rw2 = fma(xw, xw, yw * yw);
  if ((!(P.flags & SART_CF_IGNORE_DET_WINDOW) && rw2 > P.radiusWindow2) || fabs(xw) > P.chipCX || fabs(yw) > P.chipCY) {
    out.windowMiss = true; out.wPost = 0.0; out.x = out.y = out.r = 0.0; out.bin = -1;
    sink.hit(out);
    return;
  }
  out.windowMiss = false;
  // ================= strongback strips rt:2149-2185
  double post = 1.0;
  {
    // strips at (i + 0.5) d + i w < |y| < (i + 0.5) d + (i + 1) w, i = 0 .. nStripHalf-1  (closed form of the loop)
    const double yt = fabs(yw * P.cosTheta - xw * P.sinTheta);
    int sb = 2;
    if (P.nStripHalf > 0) {
      const double pitch = P.stripDist + P.stripWidth;
      const double u = yt - 0.5 * P.stripDist;
      const double fi = floor(u * P.invStripPitch);
      const double off = u - fi * pitch;
      sb = (u > 0.0 && fi < double(P.nStripHalf) && off > 0.0 && off < P.stripWidth) ? 1 : 0;
    }
    const float tw = sb == 1 ? el.Tstrongback : (sb == 0 ? el.Twindow : 0.f);
    const bool ignoreWin = (P.flags & SART_CF_IGNORE_DET_WINDOW) != 0;
    if (!ignoreWin) post *= double(tw);
    if (el.sbExp != 0) {   // rare: an energy at which a Henke grid clamps, or soft X-rays on a strip (fast_params.h: EnergyLUT)
      const int cl = el.sbExp >> 16;
      out.clamped |= (cl & (sb == 1 ? kLutClampStrongback : (sb == 0 ? kLutClampWindow : 0)) | (cl & kLutClampGas)) != 0;
      const int ex = (el.sbExp << 16) >> 16;
      if (!ignoreWin && sb == 1 && ex != 0)
        post = __hiloint2double(__double2hiint(post) + ex * (1 << 20), __double2loint(post));
    }
  }
  if (!(P.flags & SART_CF_IGNORE_GAS_ABS)) post *= double(el.Agas);
  if (!(P.flags & SART_CF_XRAY_TEST)) post *= double(P.exposure);
  out.wPost = post;
  out.r = rw2 > 1e-30 ? rw2 * rsqrt_nr(rw2) : 0.0;
  out.x = -xw + P.chipCX;
  out.y = yw + P.chipCY;
  // prepareHeatmap rt:839-842
  const int cx = int(floor(out.x * P.invBinX)), cy = int(floor(out.y * P.invBinY));
  out.bin = (cx >= 0 && cx < SART_IMAGE_BINS && cy >= 0 && cy < SART_IMAGE_BINS) ? cy * SART_IMAGE_BINS + cx : -1;
  sink.hit(out);
}

template <bool kWolter, bool kFold>
__device__ __forceinline__ void trace_one(const FastParams& P, const FastTables& T, const Smem& S, uint64_t seed,
                                          uint64_t ray, double m2, RayResult& out) {
  Rec rec;
  const int code = stage_a<kWolter>(P, T, S, seed, ray, rec);
  const RetraceQueue noQueue{nullptr, nullptr, 0u, 0u};   // mode 1 has no margins: nothing is re-traced
  RecordSink<kFold> sink{out, m2, noQueue, false};
  if (code >= 0) { sink.fail(code); return; }
  stage_b<kWolter>(P, T, S, rec, sink);
}

// ---- fused kernel ---------------------------------------------------------------------------------------------
// kBands: the variant that also fills the band images B (sart_enable_band_images; fast_common.cuh: ImageSinkT). kQH: the
// variant that also fills the quantity histograms Q (sart_enable_quantity_hists; fast_common.cuh: QuantityHistSink), with
// the band images checked at run time; 1: the block's sums in shared memory, 2: in the block replicas Q.rw / Q.rw2.
template <bool kWolter, bool kBands, int kQH = 0>
__device__ __forceinline__ void fast_fused(const FastParams& P, const FastTables& T, double mAxion2, uint64_t first,
                                           uint64_t nRays, uint64_t seed, double* __restrict__ image,
                                           double* __restrict__ imageW2, sart_counters_t* __restrict__ counters,
                                           const BandImages& B, const QuantityHists& Q) {
  extern __shared__ __align__(16) unsigned char smem[];
  Smem S;
  unsigned char* tail;
  smem_layout(P, smem, S, tail);
  WarpCounters* wc = reinterpret_cast<WarpCounters*>(tail);
  smem_fill(P, T, S);
  for (int i = threadIdx.x; i < kWarpsF * int(sizeof(WarpCounters) / 4); i += kBlockF) reinterpret_cast<unsigned int*>(wc)[i] = 0u;
  unsigned int* bandN = band_counts<kBands || kQH != 0>();
  QhistSmem qs{};
  if constexpr (kQH != 0) qs = qhist_smem<kQH == 1>(tail + kWarpsF * sizeof(WarpCounters), Q);
  __syncthreads();

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  unsigned int nPassed = 0, nTill = 0, nIter = 0;
  double sumW = 0.0, sumW2 = 0.0, sumX = 0.0, sumY = 0.0, sumR = 0.0;

  const uint32_t rep = T.nImgRep > 1 ? (blockIdx.x % unsigned(T.nImgRep)) * uint32_t(T.imgRepStride) : 0u;
  auto sink = with_extras<kBands, kQH>(ImageSink{T, mAxion2, image, imageW2, rep, wc[warp], nPassed, nTill, sumW, sumW2, sumX, sumY,
                                                 sumR}, P, B, bandN, Q, qs);
  const uint64_t stride = uint64_t(gridDim.x) * kBlockF;
  for (uint64_t i = uint64_t(blockIdx.x) * kBlockF + threadIdx.x; i < nRays; i += stride) {
    ++nIter;
    Rec rec;
    const int code = stage_a<kWolter>(P, T, S, seed, first + i, rec);
    if (code >= 0) { sink.fail(code); continue; }
    stage_b<kWolter>(P, T, S, rec, sink);
  }
  // ---- block reduction and flush
  for (int o = 16; o > 0; o >>= 1) {
    nPassed += __shfl_down_sync(0xffffffffu, nPassed, o);
    nTill += __shfl_down_sync(0xffffffffu, nTill, o);
    nIter += __shfl_down_sync(0xffffffffu, nIter, o);
    sumW += __shfl_down_sync(0xffffffffu, sumW, o);
    sumW2 += __shfl_down_sync(0xffffffffu, sumW2, o);
    sumX += __shfl_down_sync(0xffffffffu, sumX, o);
    sumY += __shfl_down_sync(0xffffffffu, sumY, o);
    sumR += __shfl_down_sync(0xffffffffu, sumR, o);
  }
  __syncthreads();
  if (lane == 0) {
    sart_counters_t* c = counters;
    atomicAdd(reinterpret_cast<unsigned long long*>(&c->n_rays), (unsigned long long)nIter);
    atomicAdd(reinterpret_cast<unsigned long long*>(&c->n_exit[SART_EXIT_PASSED]), (unsigned long long)nPassed);
    atomicAdd(reinterpret_cast<unsigned long long*>(&c->n_passed), (unsigned long long)nPassed);
    atomicAdd(reinterpret_cast<unsigned long long*>(&c->n_passed_till_window), (unsigned long long)nTill);
    for (int e = 1; e < SART_N_EXIT_CODES; ++e)
      if (wc[warp].n_exit[e]) atomicAdd(reinterpret_cast<unsigned long long*>(&c->n_exit[e]), (unsigned long long)wc[warp].n_exit[e]);
    if (wc[warp].n_exit[SART_EXIT_NICKEL])
      atomicAdd(reinterpret_cast<unsigned long long*>(&c->n_hit_nickel), (unsigned long long)wc[warp].n_exit[SART_EXIT_NICKEL]);
    if (wc[warp].n_clamped) atomicAdd(reinterpret_cast<unsigned long long*>(&c->n_interp_clamped), (unsigned long long)wc[warp].n_clamped);
    atomicAdd(&c->sum_w, sumW); atomicAdd(&c->sum_w2, sumW2);
    atomicAdd(&c->sum_x, sumX); atomicAdd(&c->sum_y, sumY); atomicAdd(&c->sum_r, sumR);
  }
  if (kBands || kQH != 0) band_counts_flush(B, bandN);
  if constexpr (kQH != 0) qhist_flush<kQH == 1>(Q, qs);
}
template <bool kWolter>
__global__ void __launch_bounds__(kBlockF, 1)
k_trace_mc_fast(const __grid_constant__ FastParams P, const __grid_constant__ FastTables T, double mAxion2,
                uint64_t first, uint64_t nRays, uint64_t seed, double* __restrict__ image,
                double* __restrict__ imageW2, sart_counters_t* __restrict__ counters) {
  fast_fused<kWolter, false>(P, T, mAxion2, first, nRays, seed, image, imageW2, counters, BandImages{}, QuantityHists{});
}
template <bool kWolter>
__global__ void __launch_bounds__(kBlockF, 1)
k_trace_mc_fast_bands(const __grid_constant__ FastParams P, const __grid_constant__ FastTables T, double mAxion2,
                      uint64_t first, uint64_t nRays, uint64_t seed, double* __restrict__ image,
                      double* __restrict__ imageW2, sart_counters_t* __restrict__ counters, const __grid_constant__ BandImages B) {
  fast_fused<kWolter, true>(P, T, mAxion2, first, nRays, seed, image, imageW2, counters, B, QuantityHists{});
}
template <bool kWolter, int kQH>
__global__ void __launch_bounds__(kBlockF, 1)
k_trace_mc_fast_qhists(const __grid_constant__ FastParams P, const __grid_constant__ FastTables T, double mAxion2,
                       uint64_t first, uint64_t nRays, uint64_t seed, double* __restrict__ image,
                       double* __restrict__ imageW2, sart_counters_t* __restrict__ counters, const __grid_constant__ BandImages B,
                       const __grid_constant__ QuantityHists Q) {
  fast_fused<kWolter, false, kQH>(P, T, mAxion2, first, nRays, seed, image, imageW2, counters, B, Q);
}

// ---- fused kernel with warp-level compaction ------------------------------------------------------------------
// Stage A (sample, clip, frame, vetoes, shell) runs on 32 fresh rays per warp; the survivors are ballot-compacted into
// a per-warp shared-memory queue, and stage B (mirrors .. histogram) runs only on full batches of 32 queued rays, so
// its lanes stay busy whatever fraction of the rays the bore, pipes, spider and glass fronts remove (BabyIAXO + XMM:
// 2/3 of the launched rays never reach a mirror). Same arithmetic per ray as k_trace_mc_fast.
constexpr int kQueue = 64;
struct WarpQueue {
  double x0[kQueue], y0[kQueue], tx[kQueue], ty[kQueue], path2[kQueue];
  int meta[kQueue];   // hitLayer | eIdx << 8 | clamped << 30
};

template <bool kWolter, bool kBands>
__device__ __forceinline__ void fast_fused_compact(const FastParams& P, const FastTables& T, double mAxion2, uint64_t first,
                                                   uint64_t nRays, uint64_t seed, double* __restrict__ image,
                                                   double* __restrict__ imageW2, sart_counters_t* __restrict__ counters,
                                                   const BandImages& B) {
  extern __shared__ __align__(16) unsigned char smem[];
  Smem S;
  unsigned char* tail;
  smem_layout(P, smem, S, tail);
  WarpCounters* wc = reinterpret_cast<WarpCounters*>(tail);
  WarpQueue* queues = reinterpret_cast<WarpQueue*>(tail + kWarpsF * sizeof(WarpCounters));
  smem_fill(P, T, S);
  for (int i = threadIdx.x; i < kWarpsF * int(sizeof(WarpCounters) / 4); i += kBlockF) reinterpret_cast<unsigned int*>(wc)[i] = 0u;
  unsigned int* bandN = band_counts<kBands>();
  __syncthreads();

  constexpr unsigned kFull = 0xffffffffu;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  WarpQueue& Q = queues[warp];
  unsigned int nPassed = 0, nTill = 0, nIter = 0;
  double sumW = 0.0, sumW2 = 0.0, sumX = 0.0, sumY = 0.0, sumR = 0.0;
  const uint64_t stride = uint64_t(gridDim.x) * kBlockF;
  const uint32_t rep = T.nImgRep > 1 ? (blockIdx.x % unsigned(T.nImgRep)) * uint32_t(T.imgRepStride) : 0u;
  auto sink = with_bands<kBands>(ImageSink{T, mAxion2, image, imageW2, rep, wc[warp], nPassed, nTill, sumW, sumW2, sumX, sumY, sumR},
                                  B, bandN);
  uint64_t base = uint64_t(blockIdx.x) * kBlockF + (threadIdx.x & ~31);   // warp-uniform
  int qn = 0;                                                              // warp-uniform queue fill
  for (;;) {
    while (qn <= kQueue - 32 && base < nRays) {
      const uint64_t i = base + lane;
      base += stride;
      Rec rec;
      int code = SART_N_EXIT_CODES;
      if (i < nRays) {
        code = stage_a<kWolter>(P, T, S, seed, first + i, rec);
        ++nIter;
        if (code >= 0) atomicAdd(&wc[warp].n_exit[code], 1u);
      }
      const unsigned m = __ballot_sync(kFull, code < 0);
      if (code < 0) {
        const int pos = qn + __popc(m & ((1u << lane) - 1u));
        Q.x0[pos] = rec.x0; Q.y0[pos] = rec.y0; Q.tx[pos] = rec.tx; Q.ty[pos] = rec.ty; Q.path2[pos] = rec.path2;
        Q.meta[pos] = rec.hitLayer | (rec.eIdx << 8) | (rec.clamped ? (1 << 30) : 0);
      }
      qn += __popc(m);
    }
    if (qn == 0) break;
    __syncwarp();
    const int take = qn < 32 ? qn : 32;
    if (lane < take) {
      const int pos = qn - take + lane;
      Rec rec;
      rec.x0 = Q.x0[pos]; rec.y0 = Q.y0[pos]; rec.tx = Q.tx[pos]; rec.ty = Q.ty[pos]; rec.path2 = Q.path2[pos];
      const int meta = Q.meta[pos];
      rec.hitLayer = meta & 0xff; rec.eIdx = (meta >> 8) & 0x3fffff; rec.clamped = (meta >> 30) & 1;
      stage_b<kWolter>(P, T, S, rec, sink);
    }
    qn -= take;
    __syncwarp();
  }
  for (int o = 16; o > 0; o >>= 1) {
    nPassed += __shfl_down_sync(kFull, nPassed, o);
    nTill += __shfl_down_sync(kFull, nTill, o);
    nIter += __shfl_down_sync(kFull, nIter, o);
    sumW += __shfl_down_sync(kFull, sumW, o);
    sumW2 += __shfl_down_sync(kFull, sumW2, o);
    sumX += __shfl_down_sync(kFull, sumX, o);
    sumY += __shfl_down_sync(kFull, sumY, o);
    sumR += __shfl_down_sync(kFull, sumR, o);
  }
  __syncwarp();
  if (lane == 0) {
    sart_counters_t* c = counters;
    auto addu = [](uint64_t* p, unsigned long long v) { if (v) atomicAdd(reinterpret_cast<unsigned long long*>(p), v); };
    addu(&c->n_rays, nIter);
    addu(&c->n_exit[SART_EXIT_PASSED], nPassed);
    addu(&c->n_passed, nPassed);
    addu(&c->n_passed_till_window, nTill);
    for (int e = 1; e < SART_N_EXIT_CODES; ++e) addu(&c->n_exit[e], wc[warp].n_exit[e]);
    addu(&c->n_hit_nickel, wc[warp].n_exit[SART_EXIT_NICKEL]);
    addu(&c->n_interp_clamped, wc[warp].n_clamped);
    atomicAdd(&c->sum_w, sumW); atomicAdd(&c->sum_w2, sumW2);
    atomicAdd(&c->sum_x, sumX); atomicAdd(&c->sum_y, sumY); atomicAdd(&c->sum_r, sumR);
  }
  if (kBands) band_counts_flush(B, bandN);
}
template <bool kWolter>
__global__ void __launch_bounds__(kBlockF, 1)
k_trace_mc_fast_compact(const __grid_constant__ FastParams P, const __grid_constant__ FastTables T, double mAxion2,
                        uint64_t first, uint64_t nRays, uint64_t seed, double* __restrict__ image,
                        double* __restrict__ imageW2, sart_counters_t* __restrict__ counters) {
  fast_fused_compact<kWolter, false>(P, T, mAxion2, first, nRays, seed, image, imageW2, counters, BandImages{});
}
template <bool kWolter>
__global__ void __launch_bounds__(kBlockF, 1)
k_trace_mc_fast_compact_bands(const __grid_constant__ FastParams P, const __grid_constant__ FastTables T, double mAxion2,
                              uint64_t first, uint64_t nRays, uint64_t seed, double* __restrict__ image,
                              double* __restrict__ imageW2, sart_counters_t* __restrict__ counters,
                              const __grid_constant__ BandImages B) {
  fast_fused_compact<kWolter, true>(P, T, mAxion2, first, nRays, seed, image, imageW2, counters, B);
}

// The same with the quantity histograms QH (kQH as in fast_fused), the band images checked at run time. A copy rather than
// another instantiation of fast_fused_compact, so that the kernels built from that keep the code they had before.
template <bool kWolter, int kQH>
__global__ void __launch_bounds__(kBlockF, 1)
k_trace_mc_fast_compact_qhists(const __grid_constant__ FastParams P, const __grid_constant__ FastTables T, double mAxion2,
                               uint64_t first, uint64_t nRays, uint64_t seed, double* __restrict__ image,
                               double* __restrict__ imageW2, sart_counters_t* __restrict__ counters,
                               const __grid_constant__ BandImages B, const __grid_constant__ QuantityHists QH) {
  extern __shared__ __align__(16) unsigned char smem[];
  Smem S;
  unsigned char* tail;
  smem_layout(P, smem, S, tail);
  WarpCounters* wc = reinterpret_cast<WarpCounters*>(tail);
  WarpQueue* queues = reinterpret_cast<WarpQueue*>(tail + kWarpsF * sizeof(WarpCounters));
  smem_fill(P, T, S);
  for (int i = threadIdx.x; i < kWarpsF * int(sizeof(WarpCounters) / 4); i += kBlockF) reinterpret_cast<unsigned int*>(wc)[i] = 0u;
  unsigned int* bandN = band_counts<true>();
  const QhistSmem qs = qhist_smem<kQH == 1>(reinterpret_cast<unsigned char*>(queues + kWarpsF), QH);
  __syncthreads();

  constexpr unsigned kFull = 0xffffffffu;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  WarpQueue& Q = queues[warp];
  unsigned int nPassed = 0, nTill = 0, nIter = 0;
  double sumW = 0.0, sumW2 = 0.0, sumX = 0.0, sumY = 0.0, sumR = 0.0;
  const uint64_t stride = uint64_t(gridDim.x) * kBlockF;
  const uint32_t rep = T.nImgRep > 1 ? (blockIdx.x % unsigned(T.nImgRep)) * uint32_t(T.imgRepStride) : 0u;
  QuantityHistSink<kQH == 1> sink{{T, mAxion2, image, imageW2, rep, wc[warp], nPassed, nTill, sumW, sumW2, sumX, sumY, sumR}, P, B,
                                  bandN, band_replica(B), QH, qs, qhist_replica(QH)};
  uint64_t base = uint64_t(blockIdx.x) * kBlockF + (threadIdx.x & ~31);   // warp-uniform
  int qn = 0;                                                              // warp-uniform queue fill
  for (;;) {
    while (qn <= kQueue - 32 && base < nRays) {
      const uint64_t i = base + lane;
      base += stride;
      Rec rec;
      int code = SART_N_EXIT_CODES;
      if (i < nRays) {
        code = stage_a<kWolter>(P, T, S, seed, first + i, rec);
        ++nIter;
        if (code >= 0) atomicAdd(&wc[warp].n_exit[code], 1u);
      }
      const unsigned m = __ballot_sync(kFull, code < 0);
      if (code < 0) {
        const int pos = qn + __popc(m & ((1u << lane) - 1u));
        Q.x0[pos] = rec.x0; Q.y0[pos] = rec.y0; Q.tx[pos] = rec.tx; Q.ty[pos] = rec.ty; Q.path2[pos] = rec.path2;
        Q.meta[pos] = rec.hitLayer | (rec.eIdx << 8) | (rec.clamped ? (1 << 30) : 0);
      }
      qn += __popc(m);
    }
    if (qn == 0) break;
    __syncwarp();
    const int take = qn < 32 ? qn : 32;
    if (lane < take) {
      const int pos = qn - take + lane;
      Rec rec;
      rec.x0 = Q.x0[pos]; rec.y0 = Q.y0[pos]; rec.tx = Q.tx[pos]; rec.ty = Q.ty[pos]; rec.path2 = Q.path2[pos];
      const int meta = Q.meta[pos];
      rec.hitLayer = meta & 0xff; rec.eIdx = (meta >> 8) & 0x3fffff; rec.clamped = (meta >> 30) & 1;
      stage_b<kWolter>(P, T, S, rec, sink);
    }
    qn -= take;
    __syncwarp();
  }
  for (int o = 16; o > 0; o >>= 1) {
    nPassed += __shfl_down_sync(kFull, nPassed, o);
    nTill += __shfl_down_sync(kFull, nTill, o);
    nIter += __shfl_down_sync(kFull, nIter, o);
    sumW += __shfl_down_sync(kFull, sumW, o);
    sumW2 += __shfl_down_sync(kFull, sumW2, o);
    sumX += __shfl_down_sync(kFull, sumX, o);
    sumY += __shfl_down_sync(kFull, sumY, o);
    sumR += __shfl_down_sync(kFull, sumR, o);
  }
  __syncwarp();
  if (lane == 0) {
    sart_counters_t* c = counters;
    auto addu = [](uint64_t* p, unsigned long long v) { if (v) atomicAdd(reinterpret_cast<unsigned long long*>(p), v); };
    addu(&c->n_rays, nIter);
    addu(&c->n_exit[SART_EXIT_PASSED], nPassed);
    addu(&c->n_passed, nPassed);
    addu(&c->n_passed_till_window, nTill);
    for (int e = 1; e < SART_N_EXIT_CODES; ++e) addu(&c->n_exit[e], wc[warp].n_exit[e]);
    addu(&c->n_hit_nickel, wc[warp].n_exit[SART_EXIT_NICKEL]);
    addu(&c->n_interp_clamped, wc[warp].n_clamped);
    atomicAdd(&c->sum_w, sumW); atomicAdd(&c->sum_w2, sumW2);
    atomicAdd(&c->sum_x, sumX); atomicAdd(&c->sum_y, sumY); atomicAdd(&c->sum_r, sumR);
  }
  band_counts_flush(B, bandN);
  qhist_flush<kQH == 1>(QH, qs);
}

// ---- fused kernel, axion-mass scan ---------------------------------------------------------------------------
// Rays are traced once (lanes = rays); each ray that reaches the weight stage is then broadcast through the warp and
// weighted for all M masses at once with lanes = masses (mass lane + 32 k), so the per-mass sums live in registers of
// the lane that owns the mass and need no reduction, and the per-mass image planes are hit by distinct lanes.
template <bool kWolter, bool kSpectra, bool kRows = false>
__device__ __forceinline__ void fast_masses(const FastParams& P, const FastTables& T, const double* __restrict__ masses,
                                            int nMasses, uint64_t first, uint64_t nRays, uint64_t seed, double* __restrict__ image,
                                            double* __restrict__ imageW2, sart_counters_t* __restrict__ counters,
                                            const MassRows& R = MassRows{}) {
  extern __shared__ __align__(16) unsigned char smem[];
  Smem S;
  unsigned char* tail;
  smem_layout(P, smem, S, tail);
  WarpCounters* wc = reinterpret_cast<WarpCounters*>(tail);
  smem_fill(P, T, S);
  for (int i = threadIdx.x; i < kWarps * int(sizeof(WarpCounters) / 4); i += kBlock) reinterpret_cast<unsigned int*>(wc)[i] = 0u;
  __syncthreads();

  mass_scan_loop<SART_MAX_MASSES / 32, kSpectra, kRows>(P, T.rad, T.spec, R, masses, nMasses, first, nRays, image, imageW2, counters, wc,
                 [&](uint64_t ray, uint32_t, RayResult& r) { trace_one<kWolter, false>(P, T, S, seed, ray, 0.0, r); return false; });
}
template <bool kWolter>
__global__ void __launch_bounds__(kBlock, 2)
k_trace_mc_fast_masses(const __grid_constant__ FastParams P, const __grid_constant__ FastTables T,
                       const double* __restrict__ masses, int nMasses, uint64_t first, uint64_t nRays, uint64_t seed,
                       double* __restrict__ image, double* __restrict__ imageW2, sart_counters_t* __restrict__ counters) {
  fast_masses<kWolter, false>(P, T, masses, nMasses, first, nRays, seed, image, imageW2, counters);
}
// The same with the per-mass spectra (sart_enable_mass_spectra; T.spec holds their accumulators, see mass_spec_add).
template <bool kWolter>
__global__ void __launch_bounds__(kBlock, 2)
k_trace_mc_fast_masses_spectra(const __grid_constant__ FastParams P, const __grid_constant__ FastTables T,
                               const double* __restrict__ masses, int nMasses, uint64_t first, uint64_t nRays, uint64_t seed,
                               double* __restrict__ image, double* __restrict__ imageW2, sart_counters_t* __restrict__ counters) {
  fast_masses<kWolter, true>(P, T, masses, nMasses, first, nRays, seed, image, imageW2, counters);
}
// The same with the per-mass radial histograms and band images R (sart_enable_mass_radial_hist / _band_images; their
// mass-minor accumulators, see mass_scan_loop), and with the per-mass spectra as well (kSpectra).
template <bool kWolter, bool kSpectra>
__global__ void __launch_bounds__(kBlock, 2)
k_trace_mc_fast_masses_rows(const __grid_constant__ FastParams P, const __grid_constant__ FastTables T,
                            const double* __restrict__ masses, int nMasses, uint64_t first, uint64_t nRays, uint64_t seed,
                            double* __restrict__ image, double* __restrict__ imageW2, sart_counters_t* __restrict__ counters,
                            const __grid_constant__ MassRows R) {
  fast_masses<kWolter, kSpectra, true>(P, T, masses, nMasses, first, nRays, seed, image, imageW2, counters, R);
}

// ---- per-ray records (traceAxionWrapper in fast mode) ----------------------------------------------------------
template <bool kWolter>
__global__ void __launch_bounds__(kBlock, 2)
k_trace_mc_rays_fast(const __grid_constant__ FastParams P, const __grid_constant__ FastTables T, double mAxion2,
                     uint64_t first, uint64_t nRays, uint64_t seed, const __grid_constant__ sart_ray_out_t o) {
  extern __shared__ __align__(16) unsigned char smem[];
  Smem S;
  unsigned char* tail;
  smem_layout(P, smem, S, tail);
  smem_fill(P, T, S);
  __syncthreads();
  const uint64_t stride = uint64_t(gridDim.x) * kBlock;
  for (uint64_t i = uint64_t(blockIdx.x) * kBlock + threadIdx.x; i < nRays; i += stride) {
    RayResult r;
    trace_one<kWolter, true>(P, T, S, seed, first + i, mAxion2, r);
    // energiesAx of the rays that reach the weight stage (the f64 table value); 0 for rays clipped before
    const double energy = r.code < 0 ? (P.testXray ? double(P.srcEnergy) : fmax(__ldg(T.energies + r.eIdx), 0.03)) : 0.0;
    store_record(P, o, i, r, mAxion2, energy);
  }
}

size_t smem_bytes(const FastParams& P, int nWarps = kWarps) {
  return align16(size_t(P.nShells) * sizeof(ShellFast)) + size_t(thr_pitch(P.nRadii)) * 4 + size_t(kRadGuide) * 2 +
         align16(size_t(P.nShellGuide)) + size_t(nWarps) * sizeof(WarpCounters);
}

}  // namespace fast

cudaError_t launch_mc_image_fast(const fast::FastParams& P, const fast::FastTables& T, double mAxion, uint64_t first,
                                 uint64_t nRays, uint64_t seed, double* image, double* imageW2,
                                 sart_counters_t* counters, int smCount, bool compact, cudaStream_t s, const BandImages& bands,
                                 const QuantityHists& qh) {
  if (nRays == 0) return cudaSuccess;
  const bool wolter = launch_variant(P, T).wolter;
  const size_t smem = fast::smem_bytes(P, fast::kWarpsF) + (compact ? fast::kWarpsF * sizeof(fast::WarpQueue) : 0);
  auto run_smem = [&](size_t sm, auto kern, auto... extra) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(sm));
    if (e != cudaSuccess) return e;
    unsigned grid = 0;
    if ((e = grid_size(kern, fast::kBlockF, sm, nRays, smCount, 0, &grid)) != cudaSuccess) return e;
    kern<<<grid, fast::kBlockF, sm, s>>>(P, T, mAxion * mAxion, first, nRays, seed, image, imageW2, counters, extra...);
    return cudaGetLastError();
  };
  auto run = [&](auto kern, auto... bandArg) { return run_smem(smem, kern, bandArg...); };
  if (qh.w) {   // the variants with the quantity histograms, the band images checked at run time
    const bool smemSums = fast::qhist_sums_in_smem(smem, qh.entries);
    using KernQ = void (*)(fast::FastParams, fast::FastTables, double, uint64_t, uint64_t, uint64_t, double*, double*,
                           sart_counters_t*, BandImages, QuantityHists);
    // [compact][wolter][sums in shared memory]
    static const KernQ table[2][2][2] = {
        {{fast::k_trace_mc_fast_qhists<false, 2>, fast::k_trace_mc_fast_qhists<false, 1>},
         {fast::k_trace_mc_fast_qhists<true, 2>, fast::k_trace_mc_fast_qhists<true, 1>}},
        {{fast::k_trace_mc_fast_compact_qhists<false, 2>, fast::k_trace_mc_fast_compact_qhists<false, 1>},
         {fast::k_trace_mc_fast_compact_qhists<true, 2>, fast::k_trace_mc_fast_compact_qhists<true, 1>}}};
    return run_smem(smem + fast::qhist_smem_bytes(qh.entries, smemSums), table[compact ? 1 : 0][wolter ? 1 : 0][smemSums ? 1 : 0],
                    bands, qh);
  }
  if (bands.w)
    return run(compact ? (wolter ? fast::k_trace_mc_fast_compact_bands<true> : fast::k_trace_mc_fast_compact_bands<false>)
                       : (wolter ? fast::k_trace_mc_fast_bands<true> : fast::k_trace_mc_fast_bands<false>), bands);
  return run(compact ? (wolter ? fast::k_trace_mc_fast_compact<true> : fast::k_trace_mc_fast_compact<false>)
                     : (wolter ? fast::k_trace_mc_fast<true> : fast::k_trace_mc_fast<false>));
}

cudaError_t launch_mc_image_fast_masses(const fast::FastParams& P, const fast::FastTables& T, int nMasses,
                                        const double* dMasses, uint64_t first, uint64_t nRays, uint64_t seed,
                                        double* image, double* imageW2, sart_counters_t* counters, int smCount,
                                        cudaStream_t s, const MassRows& rows) {
  if (nRays == 0) return cudaSuccess;
  const size_t smem = fast::smem_bytes(P);
  const bool wolter = launch_variant(P, T).wolter;
  auto run = [&](auto kern, auto... extra) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return e;
    unsigned grid = 0;
    if ((e = grid_size(kern, fast::kBlock, smem, nRays, smCount, 0, &grid)) != cudaSuccess) return e;
    kern<<<grid, fast::kBlock, smem, s>>>(P, T, dMasses, nMasses, first, nRays, seed, image, imageW2, counters, extra...);
    return cudaGetLastError();
  };
  if (rows.rad.w || rows.band.w)
    return run(T.spec.eW ? (wolter ? fast::k_trace_mc_fast_masses_rows<true, true> : fast::k_trace_mc_fast_masses_rows<false, true>)
                         : (wolter ? fast::k_trace_mc_fast_masses_rows<true, false> : fast::k_trace_mc_fast_masses_rows<false, false>),
               rows);
  return run(T.spec.eW ? (wolter ? fast::k_trace_mc_fast_masses_spectra<true> : fast::k_trace_mc_fast_masses_spectra<false>)
                       : (wolter ? fast::k_trace_mc_fast_masses<true> : fast::k_trace_mc_fast_masses<false>));
}

cudaError_t launch_mc_rays_fast(const fast::FastParams& P, const fast::FastTables& T, double mAxion, uint64_t first,
                                uint64_t nRays, uint64_t seed, const sart_ray_out_t& o, int smCount, cudaStream_t s) {
  if (nRays == 0) return cudaSuccess;
  const size_t smem = fast::smem_bytes(P);
  auto kern = launch_variant(P, T).wolter ? fast::k_trace_mc_rays_fast<true> : fast::k_trace_mc_rays_fast<false>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
  if (e != cudaSuccess) return e;
  unsigned grid = 0;
  if ((e = grid_size(kern, fast::kBlock, smem, nRays, smCount, 2, &grid)) != cudaSuccess) return e;
  kern<<<grid, fast::kBlock, smem, s>>>(P, T, mAxion * mAxion, first, nRays, seed, o);
  return cudaGetLastError();
}

}  // namespace sart
