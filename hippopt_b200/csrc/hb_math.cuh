// hb_math.cuh -- scalar/dual arithmetic and 3-vector helpers shared by the kernels.
//
// The kinematics kernel runs one adjoint (reverse) sweep over the tree per lane.  With T = double the
// sweep yields one Jacobian row per lane; with T = Dual (value + one tangent) the same code yields one
// column of the Lagrangian Hessian per lane (forward-over-reverse).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace hb {

// D (8 x 8) = A (8 x 4, row) B (4 x 8, col) + C on the fp64 tensor cores.  Fragments (PTX ISA, mma.m8n8k4 .f64):
// a: row lane / 4, column lane % 4;  b: row lane % 4, column lane / 4;  c, d: row lane / 4, columns 2 (lane % 4) + {0, 1}.
__device__ __forceinline__ void dmma_m8n8k4(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

struct Dual {
  double v, d;
};

__host__ __device__ __forceinline__ Dual mkdual(double v, double d) {
  Dual r;
  r.v = v;
  r.d = d;
  return r;
}
__device__ __forceinline__ Dual operator+(Dual a, Dual b) { return mkdual(a.v + b.v, a.d + b.d); }
__device__ __forceinline__ Dual operator-(Dual a, Dual b) { return mkdual(a.v - b.v, a.d - b.d); }
__device__ __forceinline__ Dual operator*(Dual a, Dual b) { return mkdual(a.v * b.v, fma(a.v, b.d, a.d * b.v)); }
__device__ __forceinline__ Dual operator+(Dual a, double b) { return mkdual(a.v + b, a.d); }
__device__ __forceinline__ Dual operator+(double a, Dual b) { return mkdual(a + b.v, b.d); }
__device__ __forceinline__ Dual operator-(Dual a, double b) { return mkdual(a.v - b, a.d); }
__device__ __forceinline__ Dual operator-(double a, Dual b) { return mkdual(a - b.v, -b.d); }
__device__ __forceinline__ Dual operator*(Dual a, double b) { return mkdual(a.v * b, a.d * b); }
__device__ __forceinline__ Dual operator*(double a, Dual b) { return mkdual(a * b.v, a * b.d); }
__device__ __forceinline__ Dual operator-(Dual a) { return mkdual(-a.v, -a.d); }
__device__ __forceinline__ Dual operator/(Dual a, Dual b) {
  double q = a.v / b.v;
  return mkdual(q, (a.d - q * b.d) / b.v);
}
__device__ __forceinline__ Dual operator/(double a, Dual b) {
  double q = a / b.v;
  return mkdual(q, -q * b.d / b.v);
}
__device__ __forceinline__ Dual dsqrt(Dual a) {
  double s = sqrt(a.v);
  return mkdual(s, a.d / (2.0 * s));
}
__device__ __forceinline__ double dsqrt(double a) { return sqrt(a); }

// make a T from (value, tangent); the tangent is dropped for T = double
template <class T>
__device__ __forceinline__ T mk(double v, double d);
template <>
__device__ __forceinline__ double mk<double>(double v, double) {
  return v;
}
template <>
__device__ __forceinline__ Dual mk<Dual>(double v, double d) {
  return mkdual(v, d);
}
__device__ __forceinline__ double prim(double a) { return a; }
__device__ __forceinline__ double prim(Dual a) { return a.v; }
__device__ __forceinline__ double tang(double) { return 0.0; }
__device__ __forceinline__ double tang(Dual a) { return a.d; }

template <class T>
struct V3 {
  T x, y, z;
};
typedef V3<double> D3;

template <class T>
__device__ __forceinline__ V3<T> v3(T x, T y, T z) {
  V3<T> r;
  r.x = x;
  r.y = y;
  r.z = z;
  return r;
}
template <class T>
__device__ __forceinline__ V3<T> vzero() {
  return v3<T>(mk<T>(0.0, 0.0), mk<T>(0.0, 0.0), mk<T>(0.0, 0.0));
}
template <class A, class B>
struct Prom {
  typedef Dual type;
};
template <>
struct Prom<double, double> {
  typedef double type;
};

template <class A, class B>
__device__ __forceinline__ V3<typename Prom<A, B>::type> operator+(V3<A> a, V3<B> b) {
  return v3<typename Prom<A, B>::type>(a.x + b.x, a.y + b.y, a.z + b.z);
}
template <class A, class B>
__device__ __forceinline__ V3<typename Prom<A, B>::type> operator-(V3<A> a, V3<B> b) {
  return v3<typename Prom<A, B>::type>(a.x - b.x, a.y - b.y, a.z - b.z);
}
template <class A>
__device__ __forceinline__ V3<A> operator-(V3<A> a) {
  return v3<A>(-a.x, -a.y, -a.z);
}
template <class A, class B>
__device__ __forceinline__ V3<typename Prom<A, B>::type> cross(V3<A> a, V3<B> b) {
  return v3<typename Prom<A, B>::type>(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
template <class A, class B>
__device__ __forceinline__ typename Prom<A, B>::type dot(V3<A> a, V3<B> b) {
  return a.x * b.x + a.y * b.y + a.z * b.z;
}
template <class A, class B>
__device__ __forceinline__ V3<typename Prom<A, B>::type> scale(A s, V3<B> a) {
  return v3<typename Prom<A, B>::type>(s * a.x, s * a.y, s * a.z);
}
// acc + a x b and acc - a x b with two fused multiply-adds per component (a cross product followed by an addition is
// three operations per component: the multiply-add contraction only sees one product at a time)
__device__ __forceinline__ V3<double> cadd(V3<double> acc, V3<double> a, V3<double> b) {
  return v3<double>(fma(a.y, b.z, fma(-a.z, b.y, acc.x)), fma(a.z, b.x, fma(-a.x, b.z, acc.y)),
                    fma(a.x, b.y, fma(-a.y, b.x, acc.z)));
}
__device__ __forceinline__ V3<double> csub(V3<double> acc, const double* I, V3<double> a);  // acc - I a (symmetric I)
// acc + s v
__device__ __forceinline__ V3<double> sadd(V3<double> acc, double s, V3<double> v) {
  return v3<double>(fma(s, v.x, acc.x), fma(s, v.y, acc.y), fma(s, v.z, acc.z));
}
// combine a primal vector and a tangent vector into a V3<T>
template <class T>
__device__ __forceinline__ V3<T> lift(D3 p, D3 t) {
  return v3<T>(mk<T>(p.x, t.x), mk<T>(p.y, t.y), mk<T>(p.z, t.z));
}
__device__ __forceinline__ D3 ld3(const double* p) { return v3<double>(p[0], p[1], p[2]); }
__device__ __forceinline__ void st3(double* p, D3 a) {
  p[0] = a.x;
  p[1] = a.y;
  p[2] = a.z;
}
// symmetric 3x3 (xx, xy, xz, yy, yz, zz) times vector
__device__ __forceinline__ D3 symmul(const double* I, D3 a) {
  return v3<double>(I[0] * a.x + I[1] * a.y + I[2] * a.z, I[1] * a.x + I[3] * a.y + I[4] * a.z,
                    I[2] * a.x + I[4] * a.y + I[5] * a.z);
}
__device__ __forceinline__ V3<double> csub(V3<double> acc, const double* I, V3<double> a) {
  return v3<double>(fma(-I[2], a.z, fma(-I[1], a.y, fma(-I[0], a.x, acc.x))),
                    fma(-I[4], a.z, fma(-I[3], a.y, fma(-I[1], a.x, acc.y))),
                    fma(-I[5], a.z, fma(-I[4], a.y, fma(-I[2], a.x, acc.z))));
}
// row-major 3x3 times vector
__device__ __forceinline__ D3 matvec(const double* R, D3 a) {
  return v3<double>(R[0] * a.x + R[1] * a.y + R[2] * a.z, R[3] * a.x + R[4] * a.y + R[5] * a.z,
                    R[6] * a.x + R[7] * a.y + R[8] * a.z);
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

}  // namespace hb
