// std_sort.cuh -- libstdc++'s std::sort (bits/stl_algo.h, bits/stl_heap.h), restated step for step so that a device thread puts
// elements that compare equal in exactly the order g++'s std::sort does. Feature_detector::detect sorts its grid corners with
// the unstable std::sort on a score-only comparator (ref: src/Feature_detection.cpp:111, include/Feature_detection.h:29-32):
// when scores tie, introsort's pivot choices decide which corner the mask walk meets first (SURVEY Q7), and a stable sort
// selects other features.
//   __introsort_loop      : partitions while a range is longer than _S_threshold = 16, depth limit 2 * floor(log2 n); the
//                           recursion on the right part is an explicit stack (the parts are disjoint, so order is immaterial)
//   pivot                 : __move_median_to_first(first, first + 1, mid, last - 1) + __unguarded_partition(first + 1, last, first)
//   depth limit reached   : __partial_sort(first, last, last) = __heap_select (= __make_heap) + __sort_heap
//   __final_insertion_sort: guarded insertion sort of the first 16, unguarded linear inserts for the rest
// __host__ __device__ so that the CPU suite compares it with g++'s std::sort without a GPU.
#pragma once

#if defined(__CUDACC__)
#define DSDTM_SORT_HD __host__ __device__ __forceinline__
#else
#define DSDTM_SORT_HD inline
#endif

namespace dsdtm {
namespace stdsort {

static const int kThreshold = 16;   // _S_threshold

template <class T>
DSDTM_SORT_HD void iter_swap(T* a, T* b) { const T t = *a; *a = *b; *b = t; }

template <class T, class Less>
DSDTM_SORT_HD void move_median_to_first(T* result, T* a, T* b, T* c, Less less)
{
    if (less(*a, *b)) {
        if (less(*b, *c)) iter_swap(result, b);
        else if (less(*a, *c)) iter_swap(result, c);
        else iter_swap(result, a);
    } else if (less(*a, *c)) iter_swap(result, a);
    else if (less(*b, *c)) iter_swap(result, c);
    else iter_swap(result, b);
}

template <class T, class Less>
DSDTM_SORT_HD T* unguarded_partition(T* first, T* last, T* pivot, Less less)
{
    while (true) {
        while (less(*first, *pivot)) ++first;
        --last;
        while (less(*pivot, *last)) --last;
        if (!(first < last)) return first;
        iter_swap(first, last);
        ++first;
    }
}

template <class T, class Less>
DSDTM_SORT_HD void push_heap(T* first, long hole, long top, T value, Less less)
{
    long parent = (hole - 1) / 2;
    while (hole > top && less(first[parent], value)) {
        first[hole] = first[parent];
        hole = parent;
        parent = (hole - 1) / 2;
    }
    first[hole] = value;
}

template <class T, class Less>
DSDTM_SORT_HD void adjust_heap(T* first, long hole, long len, T value, Less less)
{
    const long top = hole;
    long child = hole;
    while (child < (len - 1) / 2) {
        child = 2 * (child + 1);
        if (less(first[child], first[child - 1])) child--;
        first[hole] = first[child];
        hole = child;
    }
    if ((len & 1) == 0 && child == (len - 2) / 2) {
        child = 2 * (child + 1);
        first[hole] = first[child - 1];
        hole = child - 1;
    }
    push_heap(first, hole, top, value, less);
}

// __partial_sort(first, last, last): __heap_select degenerates to __make_heap, then __sort_heap
template <class T, class Less>
DSDTM_SORT_HD void heap_sort(T* first, T* last, Less less)
{
    const long len = last - first;
    if (len >= 2) {
        for (long parent = (len - 2) / 2;; --parent) {
            adjust_heap(first, parent, len, first[parent], less);
            if (parent == 0) break;
        }
    }
    while (last - first > 1) {
        --last;
        const T value = *last;          // __pop_heap(first, last, last)
        *last = *first;
        adjust_heap(first, 0L, (long)(last - first), value, less);
    }
}

template <class T, class Less>
DSDTM_SORT_HD void unguarded_linear_insert(T* last, Less less)
{
    const T val = *last;
    T* next = last - 1;
    while (less(val, *next)) {
        *last = *next;
        last = next;
        --next;
    }
    *last = val;
}

template <class T, class Less>
DSDTM_SORT_HD void insertion_sort(T* first, T* last, Less less)
{
    if (first == last) return;
    for (T* i = first + 1; i != last; ++i) {
        if (less(*i, *first)) {
            const T val = *i;
            for (T* p = i; p != first; --p) *p = *(p - 1);     // move_backward(first, i, i + 1)
            *first = val;
        } else {
            unguarded_linear_insert(i, less);
        }
    }
}

DSDTM_SORT_HD int lg(long n)   // std::__lg
{
    int r = -1;
    while (n) { n >>= 1; ++r; }
    return r;
}

}  // namespace stdsort

// std::sort(a, a + n, less) with libstdc++'s exact sequence of comparisons and moves
template <class T, class Less>
DSDTM_SORT_HD void std_sort(T* a, long n, Less less)
{
    using namespace stdsort;
    if (n <= 0) return;
    struct Range { int first, last, depth; };   // offsets into a (n < 2^31)
    Range stack[64];                    // one entry per partition level: at most 2 * floor(log2 n) + 1 <= 64
    int sp = 0;
    stack[sp++] = Range{ 0, (int)n, 2 * lg(n) };
    while (sp > 0) {
        const Range r = stack[--sp];
        T* first = a + r.first;
        T* last = a + r.last;
        int depth = r.depth;
        while (last - first > kThreshold) {
            if (depth == 0) {
                heap_sort(first, last, less);
                break;
            }
            --depth;
            T* mid = first + (last - first) / 2;
            move_median_to_first(first, first + 1, mid, last - 1, less);
            T* cut = unguarded_partition(first + 1, last, first, less);
            stack[sp++] = Range{ (int)(first - a), (int)(cut - a), depth };   // the loop's own continuation, taken after the "recursion" on [cut, last)
            first = cut;
        }
    }
    if (n > kThreshold) {               // __final_insertion_sort
        insertion_sort(a, a + kThreshold, less);
        for (T* i = a + kThreshold; i != a + n; ++i) unguarded_linear_insert(i, less);
    } else {
        insertion_sort(a, a + n, less);
    }
}

}  // namespace dsdtm
