// labels_test01.cxx — the label-map setters of include/itkCuberilleImageToMeshFilter.h (SetLabelValues,
// ClearLabelValues and the getters), built against the minimal ITK stand-in (tests/itk_shim).  Two modes:
//   labels_test01 Instantiate
//       no device needed: the setters and getters instantiate and behave for every pixel type of the reference's users
//   labels_test01 LabelsTest01 <in.mha> <label> [label ...]
//       every label of an uncompressed 3-D MET_UCHAR MetaImage in one Update(), after checking that Update() refuses
//       the labels while the default projection is on; each label's part of the mesh must equal the mesh of a
//       SetLabelValue( k ) run of the same filter class, points bit for bit and cells with the ids shifted.
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <iterator>
#include <map>
#include <sstream>
#include <string>
#include <vector>

#include "itkImage.h"
#include "itkMesh.h"
#include "itkCuberilleImageToMeshFilter.h"

template <typename TPixel, typename TMeshPixel>
int Instantiate()
{
  typedef itk::CuberilleImageToMeshFilter<itk::Image<TPixel, 3>, itk::Mesh<TMeshPixel, 3> > FilterType;
  typename FilterType::Pointer f = FilterType::New();
  if ( !f->GetLabelValues().empty() || !f->GetLabelPointOffsets().empty() || !f->GetLabelCellOffsets().empty() ) { return 1; }
  std::vector<TPixel> labels;
  labels.push_back( static_cast<TPixel>( 3 ) );
  labels.push_back( static_cast<TPixel>( 1 ) );
  f->SetLabelValues( labels );
  if ( f->GetLabelValues() != labels ) { return 1; }
  f->ClearLabelValues();
  if ( !f->GetLabelValues().empty() ) { return 1; }
  f->SetLabelValues( labels );
  f->SetLabelValues( std::vector<TPixel>() );
  return f->GetLabelValues().empty() ? 0 : 1;
}

typedef unsigned char PixelType;
typedef itk::Image< PixelType, 3 > ImageType;
typedef itk::Mesh< PixelType, 3 > MeshType;
typedef itk::CuberilleImageToMeshFilter< ImageType, MeshType > CuberilleType;

static ImageType::Pointer ReadRawMetaImage( const char * filename )
{
  std::ifstream f( filename, std::ios::binary );
  if ( !f ) { throw itk::ExceptionObject( __FILE__, __LINE__, std::string( "cannot open " ) + filename ); }
  std::map<std::string, std::string> meta;
  std::string line;
  while ( std::getline( f, line ) )
    {
    const size_t eq = line.find( '=' );
    if ( eq == std::string::npos ) continue;
    std::string key = line.substr( 0, eq ), val = line.substr( eq + 1 );
    while ( !key.empty() && key[key.size() - 1] == ' ' ) key.erase( key.size() - 1 );
    while ( !val.empty() && val[0] == ' ' ) val.erase( 0, 1 );
    while ( !val.empty() && ( val[val.size() - 1] == '\r' || val[val.size() - 1] == ' ' ) ) val.erase( val.size() - 1 );
    meta[key] = val;
    if ( key == "ElementDataFile" ) break;
    }
  if ( meta["ElementDataFile"] != "LOCAL" || meta["ElementType"] != "MET_UCHAR" || meta["NDims"] != "3" || meta["CompressedData"] == "True" )
    { throw itk::ExceptionObject( __FILE__, __LINE__, "unsupported MetaImage (need 3-D uncompressed MET_UCHAR, LOCAL data)" ); }
  ImageType::SizeType size; ImageType::IndexType start; start.Fill( 0 );
  { std::istringstream ss( meta["DimSize"] ); ss >> size[0] >> size[1] >> size[2]; }
  std::vector<unsigned char> payload( ( std::istreambuf_iterator<char>( f ) ), std::istreambuf_iterator<char>() );
  const size_t n = size[0] * size[1] * size[2];
  if ( payload.size() < n ) { throw itk::ExceptionObject( __FILE__, __LINE__, "MetaImage payload too short" ); }
  ImageType::Pointer image = ImageType::New();
  ImageType::RegionType region; region.SetSize( size ); region.SetIndex( start );
  image->SetRegions( region );
  image->Allocate();
  std::copy( payload.begin(), payload.begin() + n, image->GetBufferPointer() );
  return image;
}

// the points (x, y, z per point) and the cells (ids per cell) of a mesh
static void Flatten( MeshType * mesh, std::vector<float> & points, std::vector<unsigned long> & cells )
{
  points.clear();
  cells.clear();
  for ( unsigned long i = 0; i < mesh->GetNumberOfPoints(); i++ )
    {
    const MeshType::PointType & p = mesh->GetPoints()->GetElement( i );
    for ( int a = 0; a < 3; a++ ) { points.push_back( p[a] ); }
    }
  for ( unsigned long i = 0; i < mesh->GetNumberOfCells(); i++ )
    {
    MeshType::CellType * c = 0;
    mesh->GetCell( i, c );
    for ( MeshType::CellType::PointIdConstIterator it = c->PointIdsBegin(); it != c->PointIdsEnd(); ++it ) { cells.push_back( *it ); }
    }
}

int LabelsTest01( int argc, char * argv [] )
{
  if ( argc < 3 )
    {
    std::cout << "USAGE: LabelsTest01 InputImage Label [Label ...]" << std::endl;
    return EXIT_FAILURE;
    }
  std::vector<PixelType> labels;
  for ( int i = 2; i < argc; i++ ) { labels.push_back( static_cast<PixelType>( std::atoi( argv[i] ) ) ); }
  try
    {
    ImageType::Pointer image = ReadRawMetaImage( argv[1] );
    CuberilleType::Pointer filter = CuberilleType::New();
    filter->SetInput( image );
    filter->SetLabelValues( labels );
    bool refused = false;
    try
      {
      filter->Update();
      }
    catch ( itk::ExceptionObject & err )
      {
      refused = std::string( err.what() ).find( "ProjectVerticesToIsoSurfaceOff" ) != std::string::npos;
      }
    if ( !refused )
      {
      std::cerr << "ERROR: label values with projection on were not refused" << std::endl;
      return EXIT_FAILURE;
      }
    filter->ProjectVerticesToIsoSurfaceOff();
    filter->Update();
    filter->Print( std::cout );
    std::vector<float> points;
    std::vector<unsigned long> cells;
    Flatten( filter->GetOutput(), points, cells );
    const std::vector<uint64_t> & po = filter->GetLabelPointOffsets();
    const std::vector<uint64_t> & co = filter->GetLabelCellOffsets();
    std::cout << "Mesh of " << labels.size() << " labels has " << points.size() / 3 << " vertices and " << cells.size() / 3
              << " cells" << std::endl;
    if ( po.size() != labels.size() + 1 || co.size() != labels.size() + 1 || po.back() * 3 != points.size() || co.back() * 3 != cells.size() )
      {
      std::cerr << "ERROR: the label offsets do not add up to the mesh" << std::endl;
      return EXIT_FAILURE;
      }
    for ( size_t i = 0; i < labels.size(); i++ )
      {
      CuberilleType::Pointer one = CuberilleType::New();
      one->SetInput( image );
      one->SetLabelValue( labels[i] );
      one->ProjectVerticesToIsoSurfaceOff();
      one->Update();
      std::vector<float> p1;
      std::vector<unsigned long> c1;
      Flatten( one->GetOutput(), p1, c1 );
      bool same = p1.size() == 3 * ( po[i + 1] - po[i] ) && c1.size() == 3 * ( co[i + 1] - co[i] ) &&
                  ( p1.empty() || std::memcmp( &p1[0], &points[3 * po[i]], p1.size() * sizeof( float ) ) == 0 );
      for ( size_t k = 0; same && k < c1.size(); k++ ) { same = cells[3 * co[i] + k] == c1[k] + po[i]; }
      if ( !same )
        {
        std::cerr << "ERROR: the part of label " << int( labels[i] ) << " differs from its SetLabelValue run" << std::endl;
        return EXIT_FAILURE;
        }
      }
    return EXIT_SUCCESS;
    }
  catch ( itk::ExceptionObject & err )
    {
    std::cerr << "ExceptionObject caught !" << std::endl << err << std::endl;
    return EXIT_FAILURE;
    }
}

int main( int argc, char * argv [] )
{
  if ( argc > 1 && std::string( argv[1] ) == "Instantiate" )
    {
    int bad = 0;
    bad += Instantiate<unsigned char, unsigned char>();
    bad += Instantiate<signed char, float>();
    bad += Instantiate<unsigned short, unsigned short>();
    bad += Instantiate<short, double>();
    bad += Instantiate<unsigned int, float>();
    bad += Instantiate<int, int>();
    bad += Instantiate<float, float>();
    bad += Instantiate<double, double>();
    return bad;
    }
  if ( argc > 1 && std::string( argv[1] ) == "LabelsTest01" ) { return LabelsTest01( argc - 1, argv + 1 ); }
  std::cout << "USAGE: " << argv[0] << " Instantiate | LabelsTest01 <in.mha> <label> [label ...]" << std::endl;
  return EXIT_FAILURE;
}
