// Regenerates tests/golden/transvoxel_tables.bin from a checkout of the reference
// (-DVXB_TABLES_INL="<path>/src/Transvoxel.inl", included, never copied into this repo):
//
//   g++ -O1 -w -DVXB_TABLES_INL='"<reference>/src/Transvoxel.inl"' tools/gen_tables.cpp -o gen_tables
//   ./gen_tables > tests/golden/transvoxel_tables.bin
//
// The file holds the Transvoxel look-up tables re-packed for the device (byte/ushort arrays, fixed strides,
// little endian), in the order and sizes of voxels_b200/build.py TABLES_LAYOUT; build.py turns it into the
// C header the kernels and the CPU restatement include (build/gen/vxb_tables_data.h).
#include <cstdio>
#include <cstdint>
#include VXB_TABLES_INL

static void emit8(const unsigned char* data, size_t count)
{
	fwrite(data, 1, count, stdout);
}

static void emit16(const unsigned short* data, size_t count)
{
	for (size_t i = 0; i < count; ++i) { putchar(data[i] & 0xFF); putchar(data[i] >> 8); }
}

int main()
{
	emit8(regularCellClass, 256);

	unsigned char reg[16 * 16];
	for (int c = 0; c < 16; ++c) {
		reg[c * 16] = regularCellData[c].geometryCounts;
		for (int i = 0; i < 15; ++i) reg[c * 16 + 1 + i] = regularCellData[c].vertexIndex[i];
	}
	emit8(reg, sizeof(reg));
	emit16(&regularVertexData[0][0], 256 * 12);

	emit8(transitionCellClass, 512);
	unsigned char trans[56 * 40];
	for (int c = 0; c < 56; ++c) {
		for (int i = 0; i < 40; ++i) trans[c * 40 + i] = 0;
		trans[c * 40] = (unsigned char)transitionCellData[c].geometryCounts;
		for (int i = 0; i < 36; ++i) trans[c * 40 + 1 + i] = transitionCellData[c].vertexIndex[i];
	}
	emit8(trans, sizeof(trans));
	emit8(transitionCornerData, 13);
	emit16(&transitionVertexData[0][0], 512 * 12);
	return 0;
}
