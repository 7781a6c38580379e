// Stage plan of a voice program: where dsp/bank_kernel_st.cuh cuts it (pure compile-time type computation; also compiled for the
// host by the emulation harness tests/cpp/device_emul.cpp, which runs the stages back to back to check that the cut keeps every bit).
//
// The program is flattened along its Pipe spine; `Binop` / `Stack` whose LEFT operand carries the heavy leaf are re-associated with
// explicit pass-through channels
//     Binop<K, Pipe<A, M>, Y>  ==  Stack<A, MultiPass<Y::IN>>  >>  Stack<M, MultiPass<Y::IN>>  >>  Binop<K, MultiPass<M::OUT>, Y>
// (the depth-first order of the leaves — and therefore the parameter / state / uniform word layout — is unchanged; only the left
// operand, because the words of the right one must stay behind it), and consecutive light segments are merged into one stage.
#pragma once
#include "nodes.cuh"

namespace fdsp {

// ------------------------------------------------------------------ type lists
template <class... S> struct Chain { static constexpr int N = (int)sizeof...(S); };
template <class A, class B> struct Cat;
template <class... A, class... B> struct Cat<Chain<A...>, Chain<B...>> { typedef Chain<A..., B...> type; };
template <int I, class C> struct ChainAt;
template <class H, class... T> struct ChainAt<0, Chain<H, T...>> { typedef H type; };
template <int I, class H, class... T> struct ChainAt<I, Chain<H, T...>> { typedef typename ChainAt<I - 1, Chain<T...>>::type type; };
template <class C, class Acc = Chain<>> struct Rev { typedef Acc type; };
template <class H, class... T, class... A> struct Rev<Chain<H, T...>, Chain<A...>> { typedef typename Rev<Chain<T...>, Chain<H, A...>>::type type; };
template <bool B, class T, class F> struct Sel { typedef T type; };
template <class T, class F> struct Sel<false, T, F> { typedef F type; };

// ------------------------------------------------------------------ which leaves get a warp of their own
// serial recurrences with a transcendental in the loop: the per-sample latency of the whole voice is theirs
template <class G> struct IsHeavyLeaf { static constexpr bool value = false; };
template <int N> struct IsHeavyLeaf<Moog<N>> { static constexpr bool value = true; };
template <int FB, int M, int N> struct IsHeavyLeaf<NlBiquad<FB, M, 2, N>> { static constexpr bool value = true; };   // tanh-shaped feedback biquads
template <int N> struct IsHeavyLeaf<Dsf<N>> { static constexpr bool value = true; };

template <class G> struct SpineHeavy { static constexpr bool value = IsHeavyLeaf<G>::value; };
template <class X, class Y> struct SpineHeavy<Pipe<X, Y>> { static constexpr bool value = SpineHeavy<X>::value || SpineHeavy<Y>::value; };
template <int K, class X, class Y> struct SpineHeavy<Binop<K, X, Y>> { static constexpr bool value = SpineHeavy<X>::value; };   // left operand only: word order
template <class X, class Y> struct SpineHeavy<Stack<X, Y>> { static constexpr bool value = SpineHeavy<X>::value; };

// x with N extra channels passed through beside it
template <class X, int N> struct Wrap { typedef Stack<X, MultiPass<N>> type; };
template <class X> struct Wrap<X, 0> { typedef X type; };
template <class S> struct SegHeavy { static constexpr bool value = IsHeavyLeaf<S>::value; };
template <class H, int N> struct SegHeavy<Stack<H, MultiPass<N>>> { static constexpr bool value = IsHeavyLeaf<H>::value; };

// two-operand combinators as template-template arguments
template <int K> struct BinopK { template <class A, class B> using T = Binop<K, A, B>; };
struct StackK { template <class A, class B> using T = Stack<A, B>; };

// Comb<Pipe<x1 .. xm>, Y>  ->  Wrap<x1> .. Wrap<x(m-1)>, then Comb<xm, Y>  (or  Wrap<xm>, Comb<MultiPass, Y>  when xm is the heavy leaf)
template <class C, class Comb, class Y> struct CombTail;
template <class H, class Comb, class Y> struct CombTail<Chain<H>, Comb, Y> {
  typedef typename Sel<IsHeavyLeaf<H>::value, Chain<typename Wrap<H, Y::IN>::type, typename Comb::template T<MultiPass<H::OUT>, Y>>,
                       Chain<typename Comb::template T<H, Y>>>::type type;
};
template <class H, class H2, class... T, class Comb, class Y> struct CombTail<Chain<H, H2, T...>, Comb, Y> {
  typedef typename Cat<Chain<typename Wrap<H, Y::IN>::type>, typename CombTail<Chain<H2, T...>, Comb, Y>::type>::type type;
};

template <class G, bool SPLIT = SpineHeavy<G>::value> struct Flat { typedef Chain<G> type; };
template <class X, class Y> struct Flat<Pipe<X, Y>, true> { typedef typename Cat<typename Flat<X>::type, typename Flat<Y>::type>::type type; };
template <int K, class X, class Y> struct Flat<Binop<K, X, Y>, true> { typedef typename CombTail<typename Flat<X>::type, BinopK<K>, Y>::type type; };
template <class X, class Y> struct Flat<Stack<X, Y>, true> { typedef typename CombTail<typename Flat<X>::type, StackK, Y>::type type; };

// ------------------------------------------------------------------ segments -> stages
// Stages are kept most-recent-first while grouping. MODE: 0 nothing open, 1 head is an open light stage, 2 head is a heavy stage.
// A heavy segment always starts its own stage (absorbing a tiny light stage in front of it); tiny light segments behind a heavy
// stage are absorbed by it (a pan or a gain is not worth a warp); other light segments merge with each other.
constexpr int ST_TINY = 16;
template <class Stages, int MODE, class Rest> struct Grp;
template <class Stages, int MODE> struct Grp<Stages, MODE, Chain<>> { typedef Stages type; };
template <class S, class... R> struct Grp<Chain<>, 0, Chain<S, R...>> { typedef typename Grp<Chain<S>, SegHeavy<S>::value ? 2 : 1, Chain<R...>>::type type; };
template <class H, class... St, class S, class... R> struct Grp<Chain<H, St...>, 1, Chain<S, R...>> {
  static constexpr bool heavy = SegHeavy<S>::value, absorb = heavy && Cost<H>::value <= ST_TINY;
  typedef typename Sel<heavy, typename Sel<absorb, Chain<Pipe<H, S>, St...>, Chain<S, H, St...>>::type, Chain<Pipe<H, S>, St...>>::type next;
  typedef typename Grp<next, heavy ? 2 : 1, Chain<R...>>::type type;
};
template <class H, class... St, class S, class... R> struct Grp<Chain<H, St...>, 2, Chain<S, R...>> {
  static constexpr bool heavy = SegHeavy<S>::value, absorb = !heavy && Cost<S>::value <= ST_TINY;
  typedef typename Sel<absorb, Chain<Pipe<H, S>, St...>, Chain<S, H, St...>>::type next;
  typedef typename Grp<next, heavy ? 2 : (absorb ? 2 : 1), Chain<R...>>::type type;
};

template <class C> struct ChainSum;
template <> struct ChainSum<Chain<>> { static constexpr int np = 0, ns = 0, nu = 0; };
template <class H, class... T> struct ChainSum<Chain<H, T...>> {
  static constexpr int np = H::NP + ChainSum<Chain<T...>>::np, ns = H::NS + ChainSum<Chain<T...>>::ns, nu = H::NU + ChainSum<Chain<T...>>::nu;
};
template <class C> struct ChainLinked { static constexpr bool value = true; };
template <class A, class B, class... T> struct ChainLinked<Chain<A, B, T...>> { static constexpr bool value = A::OUT == B::IN && ChainLinked<Chain<B, T...>>::value; };
template <int I, class C> struct NsBefore { static constexpr int value = 0; };
template <int I, class H, class... T> struct NsBefore<I, Chain<H, T...>> { static constexpr int value = I == 0 ? 0 : H::NS + NsBefore<(I > 0 ? I - 1 : 0), Chain<T...>>::value; };

template <class G> struct StagePlan {
  typedef typename Rev<typename Grp<Chain<>, 0, typename Flat<G>::type>::type>::type all;
  static constexpr bool usable = all::N >= 2 && all::N <= 4;
  typedef typename Sel<usable, all, Chain<G>>::type stages;
  static constexpr int K = stages::N;
  template <int I> using At = typename ChainAt<I, stages>::type;
  static_assert(ChainLinked<stages>::value, "stage arities must chain");
  static_assert(ChainSum<stages>::np == G::NP && ChainSum<stages>::ns == G::NS && ChainSum<stages>::nu == G::NU, "staging must keep the word layout");
  static_assert(ChainAt<0, stages>::type::IN == G::IN && ChainAt<K - 1, stages>::type::OUT == G::OUT, "staging must keep the program's arity");
};
template <class C> struct MidSum { static constexpr int value = 0; };
template <class A, class B, class... T> struct MidSum<Chain<A, B, T...>> { static constexpr int value = A::OUT + MidSum<Chain<B, T...>>::value; };
template <int I, class C> struct MidBefore { static constexpr int value = 0; };   // sum of OUT of stages < I
template <int I, class H, class... T> struct MidBefore<I, Chain<H, T...>> { static constexpr int value = I == 0 ? 0 : H::OUT + MidBefore<(I > 0 ? I - 1 : 0), Chain<T...>>::value; };
// floats of hand-off ring of the CTA (all K-1 boundaries)
template <class G> FDSP_HDC constexpr size_t st_hand_floats(int nt, bool mix) { return st_ring_floats(G::OUT, MidSum<typename StagePlan<G>::stages>::value, nt, mix); }

}  // namespace fdsp
