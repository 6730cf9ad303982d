// hash_table.cuh -- the open-addressing table behind the volume's block hash (block key -> pool slot) and the k-NN grids'
// cell hash (cell key -> bucket): u64 keys (kEmptyKey marks a free entry), hash_key() and linear probing over a
// power-of-two capacity, an int32 value per entry, load factor at most one half.  Every probe loop lives here.
#pragma once
#include "common.cuh"

namespace otslam {

struct HashTable {
    uint64_t* keys;      // [cap], kEmptyKey = free
    int32_t* vals;       // [cap]
    uint32_t cap_mask;   // cap - 1, cap a power of two
};

// the load-factor rule: a table of `cap` entries holds at most cap / 2 keys
__host__ inline bool hash_fits(int64_t n_entries, uint32_t cap) { return (uint64_t)n_entries * 2 <= cap; }

// read-only lookup: the key's value, or -1 when it is absent.  The loop is bounded, so a full table cannot hang a reader.
__device__ __forceinline__ int hash_find(const HashTable& t, uint64_t key) {
    uint32_t h = hash_key(key) & t.cap_mask;
    for (uint32_t probe = 0; probe <= t.cap_mask; ++probe) {
        const uint64_t k = t.keys[h];
        if (k == key) return t.vals[h];
        if (k == kEmptyKey) return -1;
        h = (h + 1) & t.cap_mask;
    }
    return -1;
}

// find or insert, safe against concurrent inserts of the same or other keys: the entry index, or -1 when the table is
// full.  A new entry's value is atomicAdd(counter, 1), and `inserted` tells the caller that this thread made it.
__device__ __forceinline__ int hash_find_or_insert(const HashTable& t, uint64_t key, int* counter, bool& inserted) {
    inserted = false;
    uint32_t h = hash_key(key) & t.cap_mask;
    for (uint32_t probe = 0; probe <= t.cap_mask; ++probe) {
        const uint64_t k = *reinterpret_cast<volatile uint64_t*>(t.keys + h);
        if (k == key) return (int)h;
        if (k == kEmptyKey) {
            const unsigned long long old = atomicCAS(reinterpret_cast<unsigned long long*>(t.keys + h),
                                                     (unsigned long long)kEmptyKey, (unsigned long long)key);
            if (old == (unsigned long long)kEmptyKey) {
                t.vals[h] = atomicAdd(counter, 1);
                inserted = true;
                return (int)h;
            }
            if (old == (unsigned long long)key) return (int)h;
        }
        h = (h + 1) & t.cap_mask;
    }
    return -1;
}

// insert (key, val).  Precondition: the keys of all concurrent inserts are distinct and absent from the table, and the
// table has room for them (hash_fits) -- the loop has no bound.
__device__ __forceinline__ void hash_insert_absent(const HashTable& t, uint64_t key, int32_t val) {
    uint32_t h = hash_key(key) & t.cap_mask;
    for (;;) {
        if (atomicCAS(reinterpret_cast<unsigned long long*>(t.keys + h), (unsigned long long)kEmptyKey, (unsigned long long)key) ==
            (unsigned long long)kEmptyKey) {
            t.vals[h] = val;
            return;
        }
        h = (h + 1) & t.cap_mask;
    }
}

}  // namespace otslam
